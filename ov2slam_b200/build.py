"""Build libov2b200.so (hand-written sm_100a CUDA + the extern "C" ABI of include/ov2b200.h).

Plain nvcc, in-tree output (ov2slam_b200/lib/), so the library travels to the GPU box with the
repo snapshot.  nvcc cross-compiles without a GPU.  No torch in the link: the ABI is plain C.
"""
from __future__ import annotations

import os
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent
CSRC = ROOT / "csrc"
LIB = ROOT / "lib"
SO = LIB / "libov2b200.so"

ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden"]

# Per-file flags.  The image kernels reproduce OpenCV's float32 operation order, so FMA
# contraction is off there (-fmad=false); the FMAs OpenCV itself issues are explicit __fmaf_rn.
SOURCES = {
    "ctx.cu": [],
    "frontend_pyr.cu": ["-fmad=false"],
    "frontend_klt.cu": ["-fmad=false"],
    "frontend_fast.cu": ["-fmad=false"],
    "frontend_desc.cu": ["-fmad=false"],
    "frontend_clahe.cu": ["-fmad=false"],
    "frontend_sscale.cu": ["-fmad=false"],
    "frontend_sad.cu": ["-fmad=false"],
    "frontend_step.cu": [],
    "ba_solver.cu": [],
    "ba_lm.cu": [],
    "ba_large.cu": [],
    "ba_comm.cu": [],
    "pnp_solver.cu": [],
    "match_map.cu": ["-fmad=false"],
}


def _nvcc() -> str:
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if c and (os.path.isabs(c) and os.path.exists(c) or not os.path.isabs(c)):
            return c
    return "nvcc"


def _newer(a: Path, b: Path) -> bool:
    return (not b.exists()) or a.stat().st_mtime > b.stat().st_mtime


def build(force: bool = False, verbose: bool = False) -> Path:
    LIB.mkdir(exist_ok=True)
    objdir = LIB / "obj"
    objdir.mkdir(exist_ok=True)
    headers = list(CSRC.glob("*.cuh")) + list(CSRC.glob("*.h")) + list((ROOT.parent / "include").glob("*.h"))
    newest_hdr = max(h.stat().st_mtime for h in headers)
    objs = []
    relink = force
    for name, extra in SOURCES.items():
        src = CSRC / name
        if not src.exists():
            continue
        obj = objdir / (name + ".o")
        if force or _newer(src, obj) or obj.stat().st_mtime < newest_hdr:
            cmd = [_nvcc(), *ARCH, *COMMON, *extra, "-c", str(src), "-o", str(obj)]
            if verbose:
                cmd.insert(1, "-Xptxas=-v")
                print(" ".join(cmd), flush=True)
            subprocess.check_call(cmd)
            relink = True
        objs.append(str(obj))
    if relink or not SO.exists():
        cmd = [_nvcc(), *ARCH, "-shared", "-o", str(SO), *objs, "-Xcompiler", "-fPIC", "-cudart", "shared"]
        if verbose:
            print(" ".join(cmd), flush=True)
        subprocess.check_call(cmd)
    return SO


def build_host_shims(verbose: bool = False) -> Path:
    """Compile the drop-in C++ classes (host/feature_extractor.cpp, host/feature_tracker.cpp) against
    the stand-in OpenCV headers and link them + a self-test driver against libov2b200.so.
    On a box with real OpenCV, compile the same .cpp files with the real headers instead."""
    host = ROOT / "host"
    build()
    objs = []
    for name in ("feature_extractor.cpp", "feature_tracker.cpp", "shim_selftest.cpp", "clahe_gpu.cpp", "clahe_selftest.cpp"):
        obj = LIB / "obj" / (name + ".o")
        src = host / name
        if _newer(src, obj) or any(_newer(h, obj) for h in host.glob("*.hpp")):
            cmd = ["g++", "-std=c++17", "-O2", "-Wall", "-fPIC", "-I", str(host / "standin"), "-c", str(src), "-o", str(obj)]
            if verbose:
                print(" ".join(cmd), flush=True)
            subprocess.check_call(cmd)
        objs.append(str(obj))
    exe = LIB / "shim_selftest"
    subprocess.check_call(["g++", "-o", str(exe), *objs[:3], "-L", str(LIB), "-lov2b200", "-lpthread",
                           "-Wl,-rpath,$ORIGIN"])
    subprocess.check_call(["g++", "-o", str(LIB / "clahe_selftest"), *objs[3:], "-L", str(LIB), "-lov2b200", "-lpthread",
                           "-Wl,-rpath,$ORIGIN"])
    build_optimizer_shim(verbose)
    return exe


def build_optimizer_shim(verbose: bool = False) -> Path:
    """Compile the drop-in Optimizer::localBA (host/optimizer_localba_gpu.cpp) against the stand-in headers that mirror
    the reference's map / optimizer interfaces (host/standin/ref) and link its self-test driver."""
    host = ROOT / "host"
    build()
    objs = []
    deps = list(host.glob("*.hpp")) + list((host / "standin" / "ref").rglob("*"))
    for name in ("optimizer_localba_gpu.cpp", "multi_view_geometry_pnp_gpu.cpp", "optimizer_selftest.cpp"):
        obj = LIB / "obj" / (name + ".o")
        src = host / name
        if _newer(src, obj) or any(d.is_file() and _newer(d, obj) for d in deps):
            cmd = ["g++", "-std=c++17", "-O2", "-Wall", "-fPIC", "-DOV2_EXTERNAL_LOOSE_FULL_BA", "-I", str(host / "standin" / "ref"),
                   "-I", str(host / "standin"), "-c", str(src), "-o", str(obj)]
            if verbose:
                print(" ".join(cmd), flush=True)
            subprocess.check_call(cmd)
        objs.append(str(obj))
    exe = LIB / "optimizer_selftest"
    subprocess.check_call(["g++", "-o", str(exe), *objs, "-L", str(LIB), "-lov2b200", "-lpthread", "-Wl,-rpath,$ORIGIN"])
    build_mapper_shim(verbose)
    build_stereo_shim(verbose)
    return exe


def build_mapper_shim(verbose: bool = False) -> Path:
    """Compile the drop-in Mapper::matchToMap (host/mapper_match_gpu.cpp) against the stand-in map headers and link its
    self-test driver."""
    host = ROOT / "host"
    build()
    objs = []
    deps = list(host.glob("*.hpp")) + list((host / "standin").rglob("*"))
    for name in ("mapper_match_gpu.cpp", "mapper_selftest.cpp"):
        obj = LIB / "obj" / (name + ".o")
        src = host / name
        if _newer(src, obj) or any(d.is_file() and _newer(d, obj) for d in deps):
            cmd = ["g++", "-std=c++17", "-O2", "-Wall", "-fPIC", "-I", str(host / "standin" / "ref"), "-I", str(host / "standin"),
                   "-c", str(src), "-o", str(obj)]
            if verbose:
                print(" ".join(cmd), flush=True)
            subprocess.check_call(cmd)
        objs.append(str(obj))
    exe = LIB / "mapper_selftest"
    subprocess.check_call(["g++", "-o", str(exe), *objs, "-L", str(LIB), "-lov2b200", "-lpthread", "-Wl,-rpath,$ORIGIN"])
    return exe


def build_stereo_shim(verbose: bool = False) -> Path:
    """Compile the drop-in MapManager::stereoMatching (host/map_manager_stereo_gpu.cpp) with the drop-in FeatureTracker against the
    stand-in map / OpenCV headers and link its self-test driver."""
    host = ROOT / "host"
    build()
    objs = []
    deps = list(host.glob("*.hpp")) + list((host / "standin").rglob("*"))
    for name in ("feature_tracker.cpp", "map_manager_stereo_gpu.cpp", "stereo_selftest.cpp"):
        obj = LIB / "obj" / (name + ".stereo.o")
        src = host / name
        if _newer(src, obj) or any(d.is_file() and _newer(d, obj) for d in deps):
            cmd = ["g++", "-std=c++17", "-O2", "-Wall", "-fPIC", "-I", str(host / "standin" / "ref"), "-I", str(host / "standin"), "-I", str(host),
                   "-c", str(src), "-o", str(obj)]
            if verbose:
                print(" ".join(cmd), flush=True)
            subprocess.check_call(cmd)
        objs.append(str(obj))
    exe = LIB / "stereo_selftest"
    subprocess.check_call(["g++", "-o", str(exe), *objs, "-L", str(LIB), "-lov2b200", "-lpthread", "-Wl,-rpath,$ORIGIN"])
    return exe


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
    print(build_host_shims(verbose=True))
