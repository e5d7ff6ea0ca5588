"""In-tree build of libirmv_b200.so (sm_100a only) with plain nvcc.

`python -m irmv_detection_b200.build` or `__graft_entry__.build()`.  The .so is git-ignored but
travels with the tree to the GPU box.
"""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libirmv_b200.so")
SOURCES = ["engine.cu", "preprocess.cu", "stem_bayer.cu", "conv_direct.cu", "conv_tc.cu", "conv_raster.cu", "dwconv.cu", "shuffle_unit.cu", "decode_nms.cu", "pnp.cu", "armors.cu", "raw_decode.cu", "awb.cu"]
NVCC_FLAGS = [
    "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
    "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr",
]


def _nvcc() -> str:
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if c and (os.path.isabs(c) and os.path.exists(c) or not os.path.isabs(c)):
            return c
    return "nvcc"


def needs_build() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES] + [
        os.path.join(CSRC, "common.cuh"),
        os.path.join(CSRC, "result_layout.h"),
        os.path.join(os.path.dirname(HERE), "include", "irmv_cabi.h"),
    ]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return LIB
    objs = []
    procs = []
    os.makedirs(os.path.join(HERE, "build"), exist_ok=True)
    for s in SOURCES:
        o = os.path.join(HERE, "build", s.replace(".cu", ".o"))
        cmd = [_nvcc(), *NVCC_FLAGS, "-c", os.path.join(CSRC, s), "-o", o]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        procs.append((s, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(o)
    failed = False
    for s, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            failed = True
            sys.stderr.write(f"--- nvcc {s} failed ---\n{out}\n")
        elif verbose or out.strip():
            sys.stderr.write(f"--- nvcc {s} ---\n{out}\n")
    if failed:
        raise RuntimeError("nvcc failed building libirmv_b200.so")
    link = [_nvcc(), "-shared", "-o", LIB, *objs, "-gencode", "arch=compute_100a,code=sm_100a",
            "-Xcompiler", "-fPIC", "-cudart", "shared"]
    r = subprocess.run(link, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout)
        raise RuntimeError("link failed for libirmv_b200.so")
    return LIB


HOST_LIB = os.path.join(HERE, "libirmv_detection.so")
DROP_IN_TEST = os.path.join(HERE, "drop_in_test")


def build_host(force: bool = False) -> str:
    """C++ drop-in classes (YoloEngine / PnPSolver with the reference signatures) + their test."""
    inc = os.path.join(os.path.dirname(HERE), "include")
    srcs = [os.path.join(CSRC, "host", "yolo_engine.cpp"), os.path.join(CSRC, "host", "pnp_solver.cpp"),
            os.path.join(CSRC, "host", "armor_extractor.cpp")]
    test_src = os.path.join(os.path.dirname(HERE), "tests", "cpp", "drop_in_test.cpp")
    deps = srcs + [test_src] + [os.path.join(inc, "irmv_detection", h) for h in os.listdir(os.path.join(inc, "irmv_detection"))]
    if not force and os.path.exists(HOST_LIB) and os.path.exists(DROP_IN_TEST) and \
            all(os.path.getmtime(d) < min(os.path.getmtime(HOST_LIB), os.path.getmtime(DROP_IN_TEST)) for d in deps) and \
            os.path.getmtime(LIB) < os.path.getmtime(HOST_LIB):
        return HOST_LIB
    os.makedirs(os.path.join(HERE, "build"), exist_ok=True)
    common = ["g++", "-O2", "-std=c++20", "-fPIC", f"-I{inc}"]
    rp = ["-Wl,-rpath,$ORIGIN", "-Wl,-rpath," + HERE]
    for cmd in (common + ["-shared", "-o", HOST_LIB, *srcs, f"-L{HERE}", "-lirmv_b200", *rp],
                common + ["-o", DROP_IN_TEST, test_src, f"-L{HERE}", "-lirmv_detection", "-lirmv_b200", "-lpthread",
                          "-Wl,-rpath," + HERE]):
        r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        if r.returncode != 0:
            sys.stderr.write(r.stdout)
            raise RuntimeError("host C++ build failed: " + " ".join(cmd))
    return HOST_LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
    print(build_host(force="--force" in sys.argv))
