"""Compile check of the drop-in C++ classes (ov2slam_b200/host/*.cpp) against the REFERENCE'S OWN HEADERS (/root/reference/include) - not
the stand-in map classes of host/standin/ref that the self-tests use.  The third-party headers the reference needs and this container
lacks are the stand-ins of this directory (Eigen: mini/, OpenCV containers: mini_cv/, PCL: mini_pcl/, Ceres: the reference tree's real
public headers + miniglog, Sophus: the reference tree's real headers).

The two drop-in headers (host/feature_extractor.hpp, host/feature_tracker.hpp) REPLACE the reference's files of the same name
(INTEGRATION.md step 2): the reference's headers include each other with quotes, which looks in their own directory first, so an
include-path order cannot substitute them.  The check therefore compiles against an overlay directory: links to every reference header
except those two, which link to the drop-ins.

Needs the original project's sources, so it is not part of the test suite: run it as `python -m oracle.ref_build.check_shims`."""
from __future__ import annotations

import os
import subprocess
from pathlib import Path

HERE = Path(__file__).resolve().parent
ROOT = HERE.parents[1]
HOST = ROOT / "ov2slam_b200" / "host"
REF = Path("/root/reference")
OVERLAY = HERE.parent / "_ref" / "overlay_include"
SHIMS = ["feature_extractor.cpp", "feature_tracker.cpp", "clahe_gpu.cpp", "optimizer_localba_gpu.cpp", "multi_view_geometry_pnp_gpu.cpp",
         "mapper_match_gpu.cpp", "map_manager_stereo_gpu.cpp"]


def available() -> bool:
    return (REF / "include").exists()


def make_overlay() -> Path:
    OVERLAY.mkdir(parents=True, exist_ok=True)
    for p in OVERLAY.iterdir():
        if p.is_symlink() or p.is_file():
            p.unlink()
    for h in (REF / "include").iterdir():
        target = HOST / h.name if h.name in ("feature_extractor.hpp", "feature_tracker.hpp") else h
        link = OVERLAY / h.name
        if link.exists() or link.is_symlink():
            if link.is_dir() and not link.is_symlink():
                continue
            link.unlink()
        os.symlink(target, link)
    for extra in ("pyr_cache.hpp", "clahe_gpu.hpp"):
        link = OVERLAY / extra
        if not link.exists():
            os.symlink(HOST / extra, link)
    return OVERLAY


def include_flags() -> list[str]:
    ceres = REF / "Thirdparty" / "ceres-solver"
    dirs = [make_overlay(), HERE / "mini_pcl", HERE / "ceres_cfg", ceres / "include", ceres / "internal" / "ceres" / "miniglog",
            HERE / "mini_cv", REF / "Thirdparty" / "Sophus", HERE / "mini", REF / "include" / "ceres_parametrization"]
    out = []
    for d in dirs:
        out += ["-I", str(d)]
    return out


def check(name: str) -> str:
    """Compiler diagnostics ('' when the shim compiles)."""
    # the shims are compiled from copies of their own directory's view: sources included by path, headers through the overlay
    r = subprocess.run(["g++", "-std=c++17", "-fsyntax-only", "-w", "-DOV2_EXTERNAL_LOOSE_FULL_BA", "-iquote", str(OVERLAY), *include_flags(),
                        "-include", "cstdint", str(HOST / name)], capture_output=True, text=True)
    return r.stderr if r.returncode else ""


if __name__ == "__main__":
    for s in SHIMS:
        e = check(s)
        print(s, "OK" if not e else "FAILED\n" + e[:2000])
