"""CPU: the laser scan output's recipe (include/d2pc_b200.h) and its shared math (csrc/scan_math.h).

- angle(y, x) against mpmath at 60 digits (special values, octant and breakpoint edges, 10^6 seeded random float
  pairs across exponents): at most 2 ulp; how many results equal glibc's atan2 bit for bit is printed.
- range(x, y) against mpmath and glibc's hypot.
- the recipe (tests/scan_ref/scan.c) against the nodelet's loop restated literally (tests/scan_ref/p2l_cloudcb.cpp, glibc
  math) on S2 scenes moved into a z-up frame and on random clouds: every bin that differs is traced to a point whose
  glibc and library math differ by at most 2 ulp.
- known answers, refused settings (d2pc_laser_scan_ranges, the host-only form of d2pc_set_laser_scan's checks), the
  LaserScan wire format of ros_lite and the node mirror's scan params."""
import ctypes as C
import math
import os
import subprocess
import sys

import mpmath as mp
import numpy as np
import pytest

import oracle
import scan_ref
import transform_ref
from conftest import ROOT
from disparity_to_point_cloud_b200 import synth

mp.mp.dps = 60
# camera optical frame (z forward, y down) -> a z-up body frame whose origin is 1 m under the camera
OPTICAL_TO_ZUP = np.float32([[0, 0, 1, 0], [-1, 0, 0, 0], [0, -1, 0, 1.0]])


def ulp_err(got: float, y: float, x: float) -> float:
    # mpmath has no signed zero: take atan2(|y|, x) and give it y's sign
    exact = mp.atan2(mp.mpf(abs(y)), mp.mpf(x)) * (-1 if math.copysign(1, y) < 0 else 1)
    if exact == 0:
        return 0.0 if got == 0 else math.inf
    return float(abs(mp.mpf(got) - exact) / math.ulp(float(exact)))


def f32(v) -> float:
    return float(np.float32(v))


def cloud(xyz) -> np.ndarray:
    xyz = np.asarray(xyz, np.float32).reshape(-1, 3)
    return np.concatenate([xyz, np.ones((len(xyz), 1), np.float32)], axis=1)


# ---- angle -------------------------------------------------------------------------------------------------------

def test_angle_special_values():
    inf, pi = math.inf, math.pi
    cases = [(0.0, 1.0, 0.0), (-0.0, 1.0, -0.0), (0.0, 0.0, 0.0), (-0.0, 0.0, -0.0), (0.0, -0.0, pi), (-0.0, -0.0, -pi),
             (0.0, -1.0, pi), (-0.0, -1.0, -pi), (0.0, -1e-45, pi), (-0.0, -3e38, -pi), (1.0, 0.0, pi / 2),
             (-1.0, -0.0, -pi / 2), (inf, inf, pi / 4), (inf, -inf, 3 * pi / 4), (-inf, inf, -pi / 4),
             (-inf, -inf, -3 * pi / 4), (1.0, inf, 0.0), (-1.0, inf, -0.0), (1.0, -inf, pi), (-1.0, -inf, -pi),
             (inf, 1.0, pi / 2), (-inf, -5.0, -pi / 2)]
    for y, x, want in cases:
        got = scan_ref.angle(y, x)
        assert got == want and math.copysign(1, got) == math.copysign(1, want), (y, x, got, want)
        assert got == math.atan2(y, x), (y, x)
    assert math.isnan(scan_ref.angle(math.nan, 1.0)) and math.isnan(scan_ref.angle(1.0, math.nan))


def edge_pairs():
    """Subnormal floats, |x| = |y|, the octant edge and the table's breakpoint edges t = (2k + 1) / 16 and k / 8."""
    sub = [f32(1e-45), f32(3e-42), f32(1.1754942e-38), f32(1.1754944e-38)]
    out = []
    for s in sub:
        out += [(s, 1.0), (1.0, s), (s, s), (s, -s), (-s, 3.0), (s, f32(2.5e-45))]
    for v in (1.0, 0.1, 3e38, 1e-30, 7.0):
        out += [(v, v), (-v, v), (v, -v), (-v, -v)]
    for j in range(17):
        t = j / 16
        for den in (1.0, 3.0, 0.7, 1e20):
            x = f32(den)
            y = f32(t * den)
            for yy in (y, float(np.nextafter(np.float32(y), np.float32(0))), float(np.nextafter(np.float32(y), np.float32(10)))):
                for sy, sx in ((1, 1), (1, -1), (-1, 1), (-1, -1)):
                    out += [(sy * yy, sx * x), (sx * x, sy * yy)]
    return out


def random_pairs(n, seed):
    rng = np.random.default_rng(seed)
    e = rng.integers(-149, 128, size=(n, 2)).astype(np.float64)
    m = rng.random((n, 2)) + 1.0
    s = np.where(rng.random((n, 2)) < 0.5, -1.0, 1.0)
    v = np.clip(m * 2.0 ** e, 0, 3.4e38) * s
    # a third of the pairs with exponents close to each other: angles everywhere, not only near the axes
    close = rng.random(n) < 1 / 3
    v[close, 1] = np.clip(v[close, 0] * rng.uniform(-4, 4, close.sum()), -3.4e38, 3.4e38)
    return v.astype(np.float32)


def test_angle_within_2_ulp_of_mpmath():
    pairs = np.float32(edge_pairs() + [tuple(p) for p in random_pairs(10 ** 6, 7100)])
    pairs = pairs[(pairs[:, 0] != 0) | (pairs[:, 1] != 0)]
    r, a = scan_ref.math_arrays(pairs[:, 1], pairs[:, 0])
    glibc = np.arctan2(pairs[:, 0].astype(np.float64), pairs[:, 1].astype(np.float64))
    worst = 0.0
    for (y, x), got in zip(pairs.astype(np.float64), a):
        worst = max(worst, ulp_err(float(got), float(y), float(x)))
    same = int(np.count_nonzero(a.view(np.uint64) == glibc.view(np.uint64)))
    print(f"angle: {len(pairs)} float pairs, max error {worst:.3f} ulp, {same} ({100 * same / len(pairs):.3f} %) "
          f"bitwise equal to glibc atan2")
    assert worst <= 2.0


def test_range_against_mpmath_and_hypot():
    pairs = np.concatenate([random_pairs(200000, 7200), np.float32(edge_pairs())])
    r, _ = scan_ref.math_arrays(pairs[:, 0], pairs[:, 1])
    worst = 0.0
    for (x, y), got in zip(pairs.astype(np.float64), r):
        exact = mp.sqrt(mp.mpf(x) ** 2 + mp.mpf(y) ** 2)
        if exact:
            worst = max(worst, float(abs(mp.mpf(got) - exact) / math.ulp(float(exact))))
    hyp = np.hypot(pairs[:, 0].astype(np.float64), pairs[:, 1].astype(np.float64))
    same = int(np.count_nonzero(r == hyp))
    print(f"range: {len(pairs)} float pairs, max error {worst:.3f} ulp, {same} bitwise equal to glibc hypot")
    assert worst <= 1.0
    assert scan_ref.rng(3.0, 4.0) == 5.0 and scan_ref.rng(-0.0, 0.0) == 0.0
    assert scan_ref.rng(math.inf, 1.0) == math.inf


# ---- the recipe against the literal nodelet loop -------------------------------------------------------------------

def outcome(x, y, z, r, a, p):
    """Per point: bin (or -1) and float range, for one choice of math."""
    f = scan_ref.fields(**p)
    pp = scan_ref.params(**p)
    n = int(np.ceil(np.float32(np.float32(f["angle_max"]) - np.float32(f["angle_min"])) / np.float32(f["angle_increment"])))
    with np.errstate(invalid="ignore"):
        ok = ~(np.isnan(x) | np.isnan(y) | np.isnan(z))
        zd = z.astype(np.float64)
        ok &= ~((zd > pp["max_height"]) | (zd < pp["min_height"]))
        ok &= ~((r < pp["range_min"]) | (r > pp["range_max"]))
        ok &= ~((a < f["angle_min"]) | (a > f["angle_max"]))
        k = np.where(ok, (a - f["angle_min"]) / f["angle_increment"], -1)
    k = np.where(ok, np.trunc(np.nan_to_num(k, nan=-1)), -1).astype(np.int64)
    k[k >= n] = -1
    return k, r.astype(np.float32)


def compare(pts, label, **p):
    pts = np.ascontiguousarray(np.asarray(pts, np.float32).reshape(-1, 4))
    ours, lit = scan_ref.scan(pts, **p), scan_ref.p2l(pts, **p)
    assert len(ours) == len(lit)
    diff = np.nonzero(ours.view(np.uint32) != lit.view(np.uint32))[0]
    x, y, z = pts[:, 0], pts[:, 1], pts[:, 2]
    r_l, a_l = scan_ref.math_arrays(x, y)
    with np.errstate(invalid="ignore"):
        r_g, a_g = np.hypot(x.astype(np.float64), y.astype(np.float64)), np.arctan2(y.astype(np.float64), x.astype(np.float64))
    k_l, f_l = outcome(x, y, z, r_l, a_l, p)
    k_g, f_g = outcome(x, y, z, r_g, a_g, p)
    moved = np.nonzero((k_l != k_g) | ((k_l >= 0) & (f_l.view(np.uint32) != f_g.view(np.uint32))))[0]
    # every point whose outcome differs sits within 2 ulp of the other math's value, i.e. on an edge
    for i in moved:
        assert abs(a_l[i] - a_g[i]) <= 2 * math.ulp(abs(a_g[i])) and abs(r_l[i] - r_g[i]) <= 2 * math.ulp(r_g[i]), i
    explained = set(k_l[moved][k_l[moved] >= 0]) | set(k_g[moved][k_g[moved] >= 0])
    assert set(diff.tolist()) <= explained, (label, sorted(set(diff.tolist()) - explained))
    print(f"{label}: {len(pts)} points, {len(ours)} bins, {len(diff)} bins differ from the literal loop, "
          f"{len(moved)} points change bin or float range between glibc and the library's math")
    return ours, diff


def zup_scene(seed, h=480, w=752):
    img = synth.s2_scene(h, w, seed)
    crop = oracle.disparity_cb_mono8(img, oracle.q_from_intrinsics())
    return np.frombuffer(transform_ref.transform(crop, OPTICAL_TO_ZUP), np.float32).reshape(-1, 4)


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_recipe_matches_the_literal_loop_on_s2_scenes(seed):
    pts = zup_scene(seed)
    ours, _ = compare(pts, f"S2 seed {seed} defaults")
    assert np.count_nonzero(np.isfinite(ours)) > 20
    compare(pts, f"S2 seed {seed} 3600 bins", angle_min=-0.7, angle_max=0.7, angle_increment=0.7 / 1800,
            min_height=0.2, max_height=1.8, range_min=0.3, range_max=12.0, use_inf=0, inf_epsilon=0.5)


def test_recipe_matches_the_literal_loop_on_random_clouds():
    rng = np.random.default_rng(7300)
    for case in range(20):
        pts = np.float32(rng.normal(0, 10 ** rng.uniform(-2, 2), (20000, 4)))
        pts[rng.random(20000) < 0.02, rng.integers(0, 3)] = np.nan
        pts[rng.random(20000) < 0.01, rng.integers(0, 3)] = np.inf
        amin = rng.uniform(-math.pi, 0)
        amax = rng.uniform(0, math.pi)
        inc = (amax - amin) / rng.choice([7, 360, 1000, 5000])
        compare(pts, f"random {case}", angle_min=amin, angle_max=amax, angle_increment=inc,
                min_height=rng.uniform(-5, 0), max_height=rng.uniform(0, 5), range_min=rng.uniform(0, 1),
                range_max=rng.uniform(5, 50), use_inf=int(rng.integers(0, 2)), inf_epsilon=rng.uniform(0, 2))


# ---- known answers -----------------------------------------------------------------------------------------------

def test_known_answers():
    n = scan_ref.scan(cloud([]))
    assert len(n) == 360 and np.all(np.isinf(n))
    # a point on +x lands in the bin of angle 0 (the middle of the default -pi..pi span)
    got = scan_ref.scan(cloud([[2.0, 0.0, 0.5]]))
    k = int((0.0 - f32(-math.pi)) / f32(math.pi / 180))
    assert got[k] == 2.0 and np.count_nonzero(np.isfinite(got)) == 1
    # a point exactly on angle_max when the span is a whole number of increments: k == n, dropped (the reference
    # would write past its vector); the same point with a half-increment more span lands in the last bin
    p = dict(angle_min=-1.0, angle_max=0.0, angle_increment=0.25)
    assert len(scan_ref.scan(cloud([]), **p)) == 4
    assert np.all(np.isinf(scan_ref.scan(cloud([[3.0, 0.0, 0.5]]), **p)))
    assert np.all(np.isinf(scan_ref.p2l(cloud([[3.0, 0.0, 0.5]]), **p)))
    got = scan_ref.scan(cloud([[3.0, 0.0, 0.5]]), angle_min=-1.0, angle_max=0.125, angle_increment=0.25)
    assert len(got) == 5 and got[4] == 3.0
    # NaN in any coordinate is skipped; inf goes on to the tests (and a point at infinite range never passes them)
    nan_inf = cloud([[math.nan, 1, 1], [1, math.nan, 1], [1, 1, math.nan], [math.inf, 0, 1], [1, 0, math.inf]])
    assert np.all(np.isinf(scan_ref.scan(nan_inf)))
    assert np.all(np.isinf(scan_ref.p2l(nan_inf)))
    # heights: the default min_height DBL_MIN drops z = 0 and z < 0; both limits are inclusive
    assert np.all(np.isinf(scan_ref.scan(cloud([[1, 0, 0.0], [1, 0, -0.0], [1, 0, -1]]))))
    assert np.isfinite(scan_ref.scan(cloud([[1, 0, 1e-45]]))).any()  # the least float above DBL_MIN
    h = dict(min_height=0.5, max_height=1.5)
    for z, kept in ((0.5, True), (1.5, True), (np.float32(0.5) - np.float32(3e-8), False), (1.5000001, False)):
        assert np.isfinite(scan_ref.scan(cloud([[1, 0, z]]), **h)).any() == kept, z
    # use_inf 0: the initial value is (float)(range_max_f + inf_epsilon)
    got = scan_ref.scan(cloud([]), use_inf=0, range_max=10.0, inf_epsilon=1.0)
    assert np.all(got == np.float32(11.0))
    got = scan_ref.scan(cloud([]), use_inf=0, range_max=0.1, inf_epsilon=1e-9)
    assert np.all(got == np.float32(float(np.float32(0.1)) + 1e-9))
    # the default n
    assert len(scan_ref.scan(cloud([]))) == 360


def test_result_is_independent_of_point_order():
    pts = zup_scene(4).copy()
    want = scan_ref.scan(pts)
    lit = scan_ref.p2l(pts)
    rng = np.random.default_rng(7400)
    for _ in range(3):
        perm = rng.permutation(len(pts))
        assert scan_ref.scan(pts[perm]).tobytes() == want.tobytes()
        assert scan_ref.p2l(pts[perm]).tobytes() == lit.tobytes()


# ---- settings: the host-only d2pc_laser_scan_ranges applies d2pc_set_laser_scan's checks ----------------------------

@pytest.fixture(scope="module")
def d2pc():
    from disparity_to_point_cloud_b200 import build
    build.build()
    import disparity_to_point_cloud_b200 as d2pc
    return d2pc


def test_ranges_for_the_defaults_and_refused_settings(d2pc):
    assert d2pc.laser_scan_ranges() == 360
    p = d2pc.laser_scan_params()
    assert (p.enabled, p.keep_cloud, p.use_inf, p.inf_epsilon) == (1, 1, 1, 1.0)
    assert (p.min_height, p.max_height, p.range_min, p.range_max) == (sys.float_info.min, sys.float_info.max, 0.0,
                                                                     sys.float_info.max)
    assert (p.angle_min, p.angle_max, p.angle_increment, p.scan_time) == (-math.pi, math.pi, math.pi / 180, 1 / 30)
    assert d2pc.laser_scan_ranges(angle_min=-1.0, angle_max=1.0, angle_increment=0.25) == 8
    assert d2pc.laser_scan_ranges(angle_min=0.5, angle_max=0.5) == 0
    for amin, amax, inc in ((-1.0, 1.0, 0.3), (-0.7, 0.7, 0.7 / 1800), (-math.pi, math.pi, 2 * math.pi / 2 ** 20)):
        want = int(np.ceil((np.float32(amax) - np.float32(amin)) / np.float32(inc)))
        assert d2pc.laser_scan_ranges(angle_min=amin, angle_max=amax, angle_increment=inc) == want
        assert len(scan_ref.scan(cloud([]), angle_min=amin, angle_max=amax, angle_increment=inc)) == want
    bad = [dict(angle_min=math.nan), dict(angle_max=math.inf), dict(angle_increment=-math.inf),
           dict(range_min=math.nan), dict(range_max=math.inf), dict(angle_increment=0.0), dict(angle_increment=-0.1),
           dict(angle_increment=1e-50), dict(angle_min=1.0, angle_max=0.5), dict(range_min=-1e-9),
           dict(range_min=2.0, range_max=1.0), dict(inf_epsilon=-1.0), dict(inf_epsilon=math.nan),
           dict(min_height=math.nan), dict(max_height=math.nan), dict(angle_increment=2 * math.pi / (2 ** 20 + 8))]
    for kw in bad:
        with pytest.raises(d2pc.D2pcError) as e:
            d2pc.laser_scan_ranges(**kw)
        assert e.value.status == -1, kw
    d2pc.laser_scan_ranges(min_height=-math.inf, max_height=math.inf)  # infinite heights are allowed
    p = d2pc.laser_scan_params()
    p.struct_size = 8
    n = C.c_uint32()
    assert d2pc.lib().d2pc_laser_scan_ranges(C.byref(p), C.byref(n)) == -1


# ---- wire format and the node mirror -------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def harness():
    from disparity_to_point_cloud_b200 import build
    build.build()
    return build.build_harness()


def test_laserscan_wire_round_trip(harness, tmp_path):
    """ros_lite's LaserScan (de)serialiser round-trips; the offline harness checks it byte for byte."""
    subprocess.run([harness, "wire", str(tmp_path / "w.bin")], check=True)


def test_node_mirror_scan_params(harness, tmp_path):
    launch = tmp_path / "s.launch"
    names = ["scan_enable", "scan_keep_cloud", "scan_min_height", "scan_max_height", "scan_angle_min",
             "scan_angle_max", "scan_angle_increment", "scan_scan_time", "scan_range_min", "scan_range_max",
             "scan_use_inf", "scan_inf_epsilon"]
    values = ["1", "0", "0.1", "2.0", "-1.0", "1.0", "0.01", "0.05", "0.2", "20", "0", "0.5"]
    params = "".join(f'    <param name="{k}" value="{v}"/>\n' for k, v in zip(names, values))
    launch.write_text('<launch>\n  <node name="n" pkg="p" type="t">\n' + params + "  </node>\n</launch>\n")
    out = subprocess.run([harness, "params", str(launch)] + names, check=True, capture_output=True, text=True).stdout
    got = dict((ln.split(" ")[0], ln.split(" ")[2]) for ln in out.splitlines())
    assert all(float(got[k]) == float(v) for k, v in zip(names, values))
    # tests/test_node_params.py checks that each lands in its settings field; nothing in the launch files turns the
    # scan on
    for name in os.listdir(os.path.join(ROOT, "launch")):
        assert "scan_" not in open(os.path.join(ROOT, "launch", name)).read()
