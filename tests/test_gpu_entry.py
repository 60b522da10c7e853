"""GPU: the driver's own entry points (__graft_entry__.smoke, a short bench.py run) exit cleanly.  The driver runs
both on a fresh B200 at round end; a stale assertion in either must show up in the GPU suite first."""
import json
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_smoke_entry_point():
    import __graft_entry__ as g
    g.smoke()


def test_bench_default_line_is_complete(tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "3",
                        "--dump-outputs", str(tmp_path)], capture_output=True, text=True, cwd=ROOT, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    for key in ("metric", "value", "unit", "n_gpus", "ms_per_step", "roofline", "cpu_baseline", "e2e", "gpu_launches",
                "clocks", "config"):
        assert key in line, key
    assert line["gpu_launches"] > 0 and line["value"] > 0
    assert 0.5 < line["roofline"]["frac"] < 1.2
    assert line["e2e"]["h2d_bytes_per_step"] > 0 and line["e2e"]["d2h_bytes_per_step"] > 0
    # --dump-outputs: the seeded sample of the last step's clouds, finite files that restate bit for bit what the oracle
    # computes for the first and the last frame of the device-resident ring (the zero disparities of the seeded input
    # reproject to +-inf / NaN)
    import numpy as np

    import bench
    import oracle
    from disparity_to_point_cloud_b200 import synth
    assert sorted(os.listdir(tmp_path)) == ["cloud.npy", "cloud_nonfinite.npy"]
    assert sum(os.path.getsize(tmp_path / f) for f in os.listdir(tmp_path)) <= 64 * 10**6
    cloud, kind = np.load(tmp_path / "cloud.npy"), np.load(tmp_path / "cloud_nonfinite.npy")
    cfg = bench.CONFIGS[4]
    w, h, ring = cfg["w"], cfg["h"], cfg["ring"]
    npts = bench.n_points(w, h)
    assert cloud.dtype == kind.dtype == np.float32 and cloud.shape == kind.shape
    assert cloud.shape[0] == ring and cloud.shape[2] == 4 and 0 < cloud.shape[1] < npts
    assert np.isfinite(cloud).all() and np.isin(kind, (0, 1, -1, 2)).all() and (kind != 0).any()
    idx = np.sort(np.random.default_rng(0).choice(npts, cloud.shape[1], replace=False))
    base = synth.s3_float(h, w, 0)
    for i in (0, ring - 1):
        want = oracle.disparity_cb_f32(np.roll(base, 131 * i + 7, axis=1), oracle.q_from_intrinsics())
        want = want.view(np.float32).reshape(npts, 4)[idx]
        want_kind = np.select([np.isposinf(want), np.isneginf(want), np.isnan(want)], [1, -1, 2], 0)
        assert np.array_equal(kind[i], want_kind), f"ring slot {i}: non-finite components"
        assert np.where(want_kind == 0, want, np.float32(0)).tobytes() == cloud[i].tobytes(), f"ring slot {i}"
