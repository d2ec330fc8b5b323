"""In-tree build of the sm_100a shared library (libdpgo_b200.so) with nvcc.

The built .so lives next to the sources (dpo_b200/lib/), is git-ignored, and travels to the GPU
box with the repo snapshot.  nvcc cross-compiles for sm_100a without a GPU.
"""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
LIB = os.path.join(LIBDIR, "libdpgo_b200.so")
SOURCES = ["dpgo_kernels.cu", "dpgo_spmv_tma.cu", "dense_inverse.cu", "dpgo_capi.cu", "dpgo_chordal.cu"]
HOST_ONLY_SOURCES = ["nd_precond.cpp"]          # host planning code inside libdpgo_b200.so (g++, OpenMP)
HEADERS = ["dpgo_device.cuh", "dpgo_kernels.cuh", "nd_precond.h", os.path.join("..", "..", "include", "dpgo_b200.h")]
HOST_ONLY_FLAGS = ["-O3", "-std=c++17", "-fPIC", "-fvisibility=hidden", "-fopenmp", "-mavx2", "-mfma", "-Wall"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
         "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden", "-Xptxas", "-v"]


def _mtime(path: str) -> float:
    return os.path.getmtime(path) if os.path.exists(path) else 0.0


def needs_build() -> bool:
    newest = max(_mtime(os.path.join(CSRC, f)) for f in SOURCES + HOST_ONLY_SOURCES + HEADERS)
    return _mtime(LIB) < newest


def build_library(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return LIB
    os.makedirs(LIBDIR, exist_ok=True)
    objdir = os.path.join(LIBDIR, "obj")
    os.makedirs(objdir, exist_ok=True)
    hdr_time = max(_mtime(os.path.join(CSRC, h)) for h in HEADERS)

    def compile_one(src: str) -> str:
        obj = os.path.join(objdir, src.replace(".cu", ".o").replace(".cpp", ".o"))
        if not force and _mtime(obj) >= max(_mtime(os.path.join(CSRC, src)), hdr_time):
            return obj
        if src.endswith(".cpp"):
            cmd = [os.environ.get("CXX", "g++")] + HOST_ONLY_FLAGS + ["-c", os.path.join(CSRC, src), "-o", obj]
        else:
            cmd = [NVCC] + FLAGS + ["-c", os.path.join(CSRC, src), "-o", obj]
        res = subprocess.run(cmd, capture_output=True, text=True)
        log = os.path.join(objdir, src + ".ptxas.log")
        with open(log, "w") as fh:
            fh.write(res.stdout + res.stderr)
        if res.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{res.stdout}\n{res.stderr}")
        if verbose:
            print(res.stderr, file=sys.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=len(SOURCES) + len(HOST_ONLY_SOURCES)) as ex:
        objs = list(ex.map(compile_one, SOURCES + HOST_ONLY_SOURCES))
    cmd = [NVCC, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-cudart", "static",
                                                  "-Xcompiler", "-fopenmp"]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError(f"link failed:\n{res.stdout}\n{res.stderr}")
    return LIB


# ---------------------------------------------------------------------------------------------------
# C++ host library (libDPGO.so: PGOAgent / QuadraticProblem / QuadraticOptimizer mirror over the C ABI)
# ---------------------------------------------------------------------------------------------------
HOST_DIR = os.path.join(HERE, "host")
HOST_SOURCES = ["DPGO_utils.cpp", "DPGO_robust.cpp", "QuadraticProblem.cpp", "QuadraticOptimizer.cpp", "PGOLogger.cpp",
                "PGOAgent.cpp", "DeviceRBCD.cpp"]
CUDA_INC = os.path.join(os.path.dirname(os.path.dirname(NVCC)), "include")     # nccl.h includes cuda_runtime.h (types only)
HOST_LIB = os.path.join(LIBDIR, "libDPGO.so")
INCLUDE = os.path.join(HERE, "..", "include")
CXX = os.environ.get("CXX", "g++")
CXXFLAGS = ["-O2", "-std=c++17", "-fPIC", "-Wall", "-Wno-sign-compare", "-Wno-unused-parameter",
            "-I", os.path.join(INCLUDE, "eigen_shim"), "-I", INCLUDE, "-I", CUDA_INC]


def build_host(force: bool = False) -> str:
    build_library()
    srcs = [os.path.join(HOST_DIR, f) for f in HOST_SOURCES]
    deps = srcs + [os.path.join(HOST_DIR, "sparse_ldl.h")]
    for root, _, files in os.walk(INCLUDE):
        deps += [os.path.join(root, f) for f in files]
    if not force and _mtime(HOST_LIB) >= max(_mtime(f) for f in deps):
        return HOST_LIB
    objdir = os.path.join(LIBDIR, "obj")
    os.makedirs(objdir, exist_ok=True)

    def compile_one(src):
        obj = os.path.join(objdir, os.path.basename(src).replace(".cpp", ".host.o"))
        res = subprocess.run([CXX] + CXXFLAGS + ["-c", src, "-o", obj], capture_output=True, text=True)
        if res.returncode != 0:
            raise RuntimeError(f"{CXX} failed for {src}:\n{res.stderr}")
        return obj

    with ThreadPoolExecutor(max_workers=6) as ex:
        objs = list(ex.map(compile_one, srcs))
    res = subprocess.run([CXX, "-shared", "-o", HOST_LIB] + objs + ["-L", LIBDIR, "-ldpgo_b200", "-lnccl", "-Wl,-rpath,$ORIGIN", "-lpthread"],
                         capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError(f"link failed:\n{res.stderr}")
    return HOST_LIB


def build_cpp_program(sources, output, defines=(), extra_includes=(), rpath=None):
    """Compile a C++ program against libDPGO.so (used for the reference's unchanged examples/tests and ours).
    rpath: where the program looks for the libraries at run time (default: this tree's lib/ by absolute path)."""
    build_host()
    os.makedirs(os.path.dirname(output), exist_ok=True)
    cmd = [CXX] + CXXFLAGS
    for inc in extra_includes:
        cmd += ["-I", inc]
    for dname in defines:
        cmd += ["-D" + dname]
    cmd += list(sources) + ["-o", output, "-L", LIBDIR, "-lDPGO", "-ldpgo_b200", "-lnccl", "-Wl,-rpath," + (rpath or LIBDIR),
                            "-lpthread"]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError(f"compile failed for {sources}:\n{res.stderr[-4000:]}")
    return output


EXAMPLES_DIR = os.path.join(HERE, "..", "examples")
EXAMPLES_BIN = os.path.join(HERE, "..", "build", "examples")


def build_examples():
    """Our own C++ drivers (examples/*.cpp) against libDPGO.so."""
    out = []
    for f in sorted(os.listdir(EXAMPLES_DIR)):
        if f.endswith(".cpp"):
            out.append(build_cpp_program([os.path.join(EXAMPLES_DIR, f)],
                                         os.path.abspath(os.path.join(EXAMPLES_BIN, f[:-4]))))
    return out


if __name__ == "__main__":
    print(build_library(force="--force" in sys.argv, verbose=True))
    print(build_host(force="--force" in sys.argv))
    for b in build_examples():
        print(b)
