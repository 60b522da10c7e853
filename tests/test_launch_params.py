"""CPU: the node mirror's launch-file loader (include/d2pc_b200/nodes.hpp, Bus::load_launch_file) keeps a value that
is not a number as a string param (transform_target_frame), and reads every number as before."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def harness():
    from disparity_to_point_cloud_b200 import build
    build.build()
    return build.build_harness()


def load(harness, launch, names):
    out = subprocess.run([harness, "params", str(launch)] + names, check=True, capture_output=True, text=True).stdout
    got = {}
    for line in out.splitlines():
        name, kind, *value = line.split(" ", 2)
        got[name] = (kind, value[0] if value else None)
    return got


def test_numbers_and_strings(harness, tmp_path):
    values = {"a": "1", "b": "-7", "c": "0.05", "d": "1e-3", "e": " 2.5 ", "f": "inf", "g": "-1.5707963",
              "frame": "/body", "frame2": "base_link", "frame3": "infrastructure", "frame4": "2abc", "empty": ""}
    launch = tmp_path / "p.launch"
    params = "".join(f'    <param name="{k}" value="{v}"/>\n' for k, v in values.items())
    launch.write_text('<launch>\n  <node name="n" pkg="p" type="t">\n' + params + "  </node>\n</launch>\n")
    got = load(harness, launch, list(values) + ["absent"])
    for k in "abcdefg":
        assert got[k][0] == "number" and float(got[k][1]) == float(values[k].strip()), k
    for k in ("frame", "frame2", "frame3", "frame4"):
        assert got[k] == ("string", values[k]), k
    assert got["empty"][0] == "string" and got["absent"] == ("missing", None)


def test_the_shipped_launch_files_read_as_numbers(harness):
    import re
    seen = 0
    for name in sorted(os.listdir(os.path.join(ROOT, "launch"))):
        path = os.path.join(ROOT, "launch", name)
        params = dict(re.findall(r'<param\s+name="([^"]*)"\s+value="([^"]*)"', open(path).read()))
        got = load(harness, path, list(params))
        for k, v in params.items():
            assert got[k][0] == "number" and float(got[k][1]) == float(v), (name, k)
        seen += len(params)
    assert seen > 0
