"""Builds the native engine (libb200tag.so) in-tree with nvcc for sm_100a."""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
LIB = os.path.join(LIBDIR, "libb200tag.so")

CU_SOURCES = ["kernels_frontend.cu", "kernels_blobs.cu", "kernels_decode.cu", "kernels_jpeg.cu", "kernels_pose.cu", "detector.cu"]
CC_SOURCES = ["pose.cc", "jpeg_host.cc"]   # host-only parts of the C ABI
HEADERS = ["dev_types.h", "kernels.h", "jpeg.h", "jpeg_core.h", "pose_core.h", "tag_families_data.h", os.path.join("..", "..", "include", "b200tag.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    # strict IEEE evaluation order: no mul+add contraction (oracle parity, DESIGN.md "Numerics")
    "-fmad=false", "-Xcompiler", "-fPIC",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.sep not in cand or os.path.exists(cand)):
            return cand
    return "nvcc"


def needs_build() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in CU_SOURCES + CC_SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def build_native(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return LIB
    os.makedirs(LIBDIR, exist_ok=True)
    objs = []
    procs = []
    for src in CU_SOURCES:
        obj = os.path.join(LIBDIR, src.replace(".cu", ".o"))
        cmd = [_nvcc(), *NVCC_FLAGS, "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    for src in CC_SOURCES:
        obj = os.path.join(LIBDIR, src.replace(".cc", ".o"))
        cmd = ["g++", "-std=c++17", "-O2", "-fPIC", "-ffp-contract=off", "-c", os.path.join(CSRC, src), "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    failed = False
    for src, pr in procs:
        out, _ = pr.communicate()
        if pr.returncode != 0 or verbose:
            sys.stderr.write(f"--- nvcc {src} ---\n{out}\n")
        failed |= pr.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed")
    cmd = [_nvcc(), "-shared", "-o", LIB, *objs, "-gencode", "arch=compute_100a,code=sm_100a", "-cudart", "static"]
    subprocess.check_call(cmd)
    return LIB


CORE_LIB = os.path.join(LIBDIR, "libapriltags_cuda_core.so")


def build_cpp_class(force: bool = False) -> str:
    """libapriltags_cuda_core.so: frc971::apriltag::GpuDetector (+ libapriltag stand-ins) over libb200tag.so."""
    inc = os.path.join(HERE, "..", "include")
    srcs = [os.path.join(CSRC, "gpu_detector.cc"), os.path.join(CSRC, "apriltag_compat.c"), os.path.join(CSRC, "gpu_detector_debug.cc")]
    deps = srcs + [os.path.join(inc, "apriltags_cuda", "apriltag_gpu.h"), os.path.join(inc, "apriltags_cuda", "reference_types.h"), os.path.join(inc, "apriltag_compat", "apriltag.h"),
                   os.path.join(inc, "b200tag.h"), LIB]
    if not force and os.path.exists(CORE_LIB) and all(os.path.getmtime(d) <= os.path.getmtime(CORE_LIB) for d in deps):
        return CORE_LIB
    flags = ["-O2", "-fPIC", "-I", inc, "-I", os.path.join(inc, "apriltag_compat"), "-I", CSRC]
    o1 = os.path.join(LIBDIR, "gpu_detector.o")
    o2 = os.path.join(LIBDIR, "apriltag_compat.o")
    o3 = os.path.join(LIBDIR, "gpu_detector_debug.o")
    subprocess.check_call(["g++", "-std=c++17", *flags, "-c", srcs[0], "-o", o1])
    subprocess.check_call(["gcc", "-std=c11", "-D_GNU_SOURCE", *flags, "-c", srcs[1], "-o", o2])
    subprocess.check_call(["g++", "-std=c++17", *flags, "-c", srcs[2], "-o", o3])
    subprocess.check_call(["g++", "-shared", "-o", CORE_LIB, o1, o2, o3, "-L", LIBDIR, "-lb200tag", "-Wl,-rpath,$ORIGIN", "-lm"])
    return CORE_LIB


def build_cpp_test() -> str:
    inc = os.path.join(HERE, "..", "include")
    exe = os.path.join(LIBDIR, "gpu_detector_test")
    src = os.path.join(HERE, "..", "tests", "cpp", "gpu_detector_test.cc")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-I", inc, "-I", os.path.join(inc, "apriltag_compat"), src, "-o", exe,
                           "-L", LIBDIR, "-lapriltags_cuda_core", "-lb200tag", "-Wl,-rpath,$ORIGIN"])
    exe2 = os.path.join(LIBDIR, "debug_accessors_test")
    src2 = os.path.join(HERE, "..", "tests", "cpp", "debug_accessors_test.cc")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-I", inc, "-I", os.path.join(inc, "apriltag_compat"), src2, "-o", exe2,
                           "-L", LIBDIR, "-lapriltags_cuda_core", "-lb200tag", "-Wl,-rpath,$ORIGIN"])
    return exe


if __name__ == "__main__":
    print(build_native(force="--force" in sys.argv, verbose="-v" in sys.argv))
    print(build_cpp_class(force="--force" in sys.argv))
    print(build_cpp_test())
