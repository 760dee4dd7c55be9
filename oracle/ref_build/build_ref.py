"""Recipe for oracle/_ref/libov2ref_residuals.so: the reference's OWN residual source (src/ceres_parametrization.cpp with its
headers, compiled where it lies under /root/reference - nothing is copied) + oracle/ref_build/residual_ref.cpp (C entry points),
with the real Sophus 1.1 and Ceres 2.0 public headers of the reference tree (Thirdparty/Sophus, Thirdparty/ceres-solver/include), against the
stand-in Eigen header of oracle/ref_build/mini (this container has no Eigen).

TEST INFRASTRUCTURE: only tests/, __graft_entry__ (build + smoke) and bench.py's CPU legs may use what this builds.
/root/reference does not exist on the GPU box: the library is built here and travels with the snapshot (oracle/_ref/ is
git-ignored, not gpurun-ignored); `build()` returns the existing file when the reference tree is absent.
"""
from __future__ import annotations

import os
import subprocess
from pathlib import Path

HERE = Path(__file__).resolve().parent
OUT = HERE.parent / "_ref" / "libov2ref_residuals.so"
REF = Path("/root/reference")
CERES = REF / "Thirdparty" / "ceres-solver"
SRC = REF / "src" / "ceres_parametrization.cpp"


def available() -> bool:
    return OUT.exists() or SRC.exists()


def build(force: bool = False) -> Path | None:
    if not os.access(SRC, os.R_OK):
        return OUT if OUT.exists() else None
    deps = [SRC, HERE / "residual_ref.cpp"] + [p for p in (HERE / "mini").rglob("*") if p.is_file()]
    if not force and OUT.exists() and all(OUT.stat().st_mtime >= d.stat().st_mtime for d in deps):
        return OUT
    OUT.parent.mkdir(parents=True, exist_ok=True)
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-w",
                           "-I", str(HERE / "ceres_cfg"), "-I", str(REF / "Thirdparty" / "ceres-solver" / "include"),
                           "-I", str(REF / "Thirdparty" / "ceres-solver" / "internal" / "ceres" / "miniglog"),
                           "-I", str(REF / "Thirdparty" / "Sophus"), "-I", str(HERE / "mini"), "-I", str(REF / "include" / "ceres_parametrization"),
                           str(SRC), str(HERE / "residual_ref.cpp"),
                           # the two Ceres base classes the cost functions derive from have out-of-line members
                           str(CERES / "internal" / "ceres" / "local_parameterization.cc"),
                           str(CERES / "internal" / "ceres" / "miniglog" / "glog" / "logging.cc"), "-I", str(CERES / "internal"),
                           "-Wl,--no-undefined", "-o", str(OUT)])
    return OUT


if __name__ == "__main__":
    print(build(force=True))
