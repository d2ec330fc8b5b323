"""Compiles the upstream project's OWN example drivers and gtest files, unchanged, against the B200 host library
(include/DPGO + libDPGO.so + libdpgo_b200.so) into oracle/_ref/bin/ ("link unchanged").

The upstream sources are not part of this repository.  They are looked for in $DPGO_REFERENCE_DIR, else in a checkout
named `reference` next to this repository; without one nothing is built and tests/test_gpu_reference_drivers.py skips.
oracle/_ref/ is a build product (git-ignored); it holds everything those tests run, so it can be copied to a GPU
machine that has no upstream checkout."""
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
OUT_DIR = os.path.join(HERE, "_ref")
BIN_DIR = os.path.join(OUT_DIR, "bin")


def reference_dir() -> str:
    return os.environ.get("DPGO_REFERENCE_DIR") or os.path.join(os.path.dirname(ROOT), "reference")


def build() -> list:
    ref = reference_dir()
    if not os.path.isdir(os.path.join(ref, "examples")):
        return []
    if ROOT not in sys.path:
        sys.path.insert(0, ROOT)
    from dpo_b200.build import INCLUDE, build_cpp_program
    # relative to the binary, so that a copy of the whole tree at another path still finds the tree's own libraries
    rpath = "$ORIGIN/../../../dpo_b200/lib"
    out = []
    for name in ("MultiRobotExample", "SingleRobotExample"):
        out.append(build_cpp_program([os.path.join(ref, "examples", name + ".cpp")], os.path.join(BIN_DIR, name),
                                     rpath=rpath))
    tests = [os.path.join(ref, "tests", f) for f in
             ("testConstruction.cpp", "testLineGraph.cpp", "testTriangleGraph.cpp", "testOptimizationThread.cpp")]
    main_cpp = os.path.join(OUT_DIR, "gtest_main.cpp")
    os.makedirs(OUT_DIR, exist_ok=True)
    with open(main_cpp, "w") as fh:
        fh.write('#define GTEST_SHIM_MAIN\n#include "gtest/gtest.h"\n')
    out.append(build_cpp_program(tests + [main_cpp], os.path.join(BIN_DIR, "testDPGO"),
                                 extra_includes=[os.path.join(INCLUDE, "gtest_shim")], rpath=rpath))
    return out


if __name__ == "__main__":
    for b in build():
        print(b)
