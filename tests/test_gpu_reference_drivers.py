"""The reference's OWN example drivers and gtest files, compiled UNCHANGED against the B200 host library
(include/DPGO + libDPGO.so + libdpgo_b200.so) by oracle/build_ref.py, run on the GPU.  The binaries are built where
a checkout of the reference exists and are carried with the tree in oracle/_ref/."""
import os
import re
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "oracle", "_ref", "bin")


def need(name):
    path = os.path.join(BIN, name)
    if not os.path.exists(path):
        pytest.skip(f"{path} not built (needs a checkout of the reference at build time, see oracle/build_ref.py)")
    return path


def test_reference_gtests_pass():
    """ref tests/testConstruction.cpp, testLineGraph.cpp, testTriangleGraph.cpp, testOptimizationThread.cpp."""
    res = subprocess.run([need("testDPGO")], capture_output=True, text=True, timeout=600)
    print(res.stdout[-3000:], res.stderr[-2000:])
    assert res.returncode == 0
    assert "5 tests ran, 0 failed" in res.stdout


@pytest.mark.parametrize("ds,expect", [("tinyGrid3D", 18.51936666), ("sphere2500", 1687.00588)])
def test_single_robot_example(ds, expect):
    """ref examples/SingleRobotExample.cpp:103 prints `Cost = 2 f(X)`; expected values from BASELINE.md section 2."""
    res = subprocess.run([need("SingleRobotExample"), os.path.join(ROOT, "data", ds + ".g2o")], capture_output=True,
                         text=True, timeout=600)
    print(res.stdout[-2000:], res.stderr[-2000:])
    assert res.returncode == 0
    m = re.search(r"Cost = ([0-9.eE+-]+)", res.stdout)
    assert m, res.stdout
    assert abs(float(m.group(1)) - expect) <= 2e-5 * expect      # cout prints 6 significant digits


def test_multi_robot_example_reproduces_shipped_trace(tmp_path):
    """ref examples/MultiRobotExample.cpp main() is hard-wired to compute(5, "torus3D", false) and writes
    ../../result/graph/NPtorus3D.txt; the reference ships that very file (first 400 lines in tests/golden/)."""
    exe = need("MultiRobotExample")
    # the driver reads ../../data/ and writes ../../result/graph/ relative to its working directory
    cwd = tmp_path / "run" / "bin"
    cwd.mkdir(parents=True)
    (tmp_path / "data").symlink_to(os.path.join(ROOT, "data"))
    (tmp_path / "result" / "graph").mkdir(parents=True)
    out = str(tmp_path / "result" / "graph" / "NPtorus3D.txt")
    res = subprocess.run([exe], cwd=str(cwd), capture_output=True, text=True, timeout=1800)
    print(res.stdout[-1500:], res.stderr[-1500:])
    assert res.returncode == 0
    got = np.loadtxt(out, delimiter=",")
    gold = np.loadtxt(os.path.join(ROOT, "tests", "golden", "NPtorus3D_head400.txt"), delimiter=",")
    k = min(len(got), len(gold))
    assert k >= 400
    assert np.max(np.abs(got[:k, 0] - gold[:k, 0]) / gold[:k, 0]) <= 5e-9
    assert np.max(np.abs(got[:k, 1] - gold[:k, 1]) / gold[:k, 1]) <= 5e-7
    # the driver stops at the first central gradient norm < 0.1: line 532 of the shipped trace (BASELINE.md)
    assert len(got) == 532
    assert got[-1, 1] < 0.1
