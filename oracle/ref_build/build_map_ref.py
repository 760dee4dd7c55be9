"""Recipe for oracle/_ref/libov2ref_map.so: the reference's OWN map and optimizer code - src/optimizer.cpp, frame.cpp, map_point.cpp,
map_manager.cpp, camera_calibration.cpp, multi_view_geometry.cpp, feature_extractor.cpp, feature_tracker.cpp, mapper.cpp, estimator.cpp (compiled where they lie,
nothing copied) - with the Ceres 2.0 objects of build_ceres_ref.py, the reference tree's Sophus, and this directory's stand-ins for what
the container lacks (Eigen: mini/, OpenCV containers: mini_cv/ with arithmetic through cv2 callbacks, PCL: mini_pcl/), plus the drivers
map_ref.cpp / fe_ref.cpp.  TEST INFRASTRUCTURE: only tests/ use what this builds."""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

from . import build_ceres_ref

HERE = Path(__file__).resolve().parent
OUTDIR = HERE.parent / "_ref"
OUT = OUTDIR / "libov2ref_map.so"
REF = Path("/root/reference")
CERES = REF / "Thirdparty" / "ceres-solver"
REF_SOURCES = ["optimizer", "frame", "map_point", "map_manager", "camera_calibration", "multi_view_geometry", "feature_extractor", "feature_tracker", "mapper",
               "estimator"]
INC = ["-I", str(HERE / "mini_pcl"), "-I", str(HERE / "ceres_cfg"), "-I", str(CERES / "include"),
       "-I", str(CERES / "internal" / "ceres" / "miniglog"), "-I", str(HERE / "mini_cv"), "-I", str(REF / "Thirdparty" / "Sophus"), "-I", str(HERE / "mini"),
       "-I", str(REF / "include"), "-I", str(REF / "include" / "ceres_parametrization")]


def available() -> bool:
    return OUT.exists() or (REF / "src" / "optimizer.cpp").exists()


def build(force: bool = False):
    if not os.access(REF / "src" / "optimizer.cpp", os.R_OK):
        return OUT if OUT.exists() else None
    if build_ceres_ref.build() is None:
        return None
    src = [REF / "src" / (n + ".cpp") for n in REF_SOURCES] + [HERE / "map_ref.cpp", HERE / "fe_ref.cpp"]
    hdrs = [p for d in ("mini", "mini_cv", "mini_pcl", "ceres_cfg") for p in (HERE / d).rglob("*") if p.is_file()]
    ceres_objs = [o for o in sorted((OUTDIR / "ceres_obj").glob("*.o")) if "ceres_ba_ref" not in o.name]
    deps = src + hdrs + ceres_objs
    if not force and OUT.exists() and all(OUT.stat().st_mtime >= d.stat().st_mtime for d in deps):
        return OUT
    objdir = OUTDIR / "map_obj"
    objdir.mkdir(parents=True, exist_ok=True)
    newest_hdr = max(h.stat().st_mtime for h in hdrs)

    def compile_one(s):
        o = objdir / (s.stem + ".o")
        if not force and o.exists() and o.stat().st_mtime >= max(s.stat().st_mtime, newest_hdr):
            return o, None
        r = subprocess.run(["g++", "-std=c++17", "-O1", "-fPIC", "-w", "-DNDEBUG", *INC, "-c", str(s), "-o", str(o)], capture_output=True, text=True)
        return o, (r.stderr if r.returncode else None)

    with ThreadPoolExecutor(max_workers=min(10, os.cpu_count() or 4)) as ex:
        results = list(ex.map(compile_one, src))
    errs = [(o, e) for o, e in results if e]
    if errs:
        for o, e in errs[:3]:
            sys.stderr.write(f"--- {o.name}\n{e[:3000]}\n")
        raise RuntimeError(f"{len(errs)} reference sources failed to compile against the stand-in headers")
    subprocess.check_call(["g++", "-shared", "-o", str(OUT), *[str(o) for o, _ in results], *[str(o) for o in ceres_objs], "-lpthread", "-Wl,--no-undefined"])
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv))
