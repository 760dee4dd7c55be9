"""Recipe for oracle/_ref/libov2ref_ceres.so: the Ceres 2.0 sources vendored in the reference tree
(/root/reference/Thirdparty/ceres-solver/internal/ceres/*.cc, compiled where they lie, nothing copied), the reference's residual
source (src/ceres_parametrization.cpp) and oracle/ref_build/ceres_ba_ref.cpp (a driver that sets a window up and solves it the way
Optimizer::localBA does), with the reference tree's own Sophus 1.1 headers, against the stand-in Eigen header of oracle/ref_build/mini
(this container has no Eigen), Ceres'
own miniglog, and a hand-written config.h for a dependency-free build (oracle/ref_build/ceres_cfg).

Not compiled: tests / benchmarks, covariance*, and three files off the DENSE_SCHUR + Levenberg-Marquardt path that need
decompositions the stand-in header lacks (dogleg_strategy.cc, polynomial.cc, line_search_direction.cc): ceres_stubs.cpp defines
their entry points as aborting stubs so that the factories link.

TEST INFRASTRUCTURE: only tests/ may use what this builds.  Built when /root/reference is present (here); the .so travels to the GPU
box with the snapshot (oracle/_ref/ is git-ignored, not gpurun-ignored).
"""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

HERE = Path(__file__).resolve().parent
OUTDIR = HERE.parent / "_ref"
OUT = OUTDIR / "libov2ref_ceres.so"
REF = Path("/root/reference")
CERES = REF / "Thirdparty" / "ceres-solver"
SKIP = ("_test", "test_util", "gmock", "benchmark", "evaluator_test_utils", "generate_", "dogleg_strategy", "polynomial",
        "line_search_direction", "covariance")
INC = ["-I", str(HERE / "ceres_cfg"), "-I", str(CERES / "include"), "-I", str(CERES / "internal"),
       "-I", str(CERES / "internal" / "ceres" / "miniglog"), "-I", str(REF / "Thirdparty" / "Sophus"), "-I", str(HERE / "mini"), "-I", str(REF / "include" / "ceres_parametrization")]
FLAGS = ["-std=c++17", "-O2", "-fPIC", "-w", "-DNDEBUG", "-DMAX_LOG_LEVEL=-1"]     # miniglog: warnings and errors only


def sources():
    src = [p for p in sorted((CERES / "internal" / "ceres").glob("*.cc")) if not any(s in p.name for s in SKIP)]
    src += [CERES / "internal" / "ceres" / "generated" / "schur_eliminator_d_d_d.cc",
            CERES / "internal" / "ceres" / "generated" / "partitioned_matrix_view_d_d_d.cc",
            CERES / "internal" / "ceres" / "miniglog" / "glog" / "logging.cc",
            REF / "src" / "ceres_parametrization.cpp", HERE / "ceres_stubs.cpp", HERE / "ceres_ba_ref.cpp"]
    return src


def available() -> bool:
    return OUT.exists() or CERES.exists()


def build(force: bool = False, verbose: bool = False):
    if not os.access(CERES, os.R_OK):
        return OUT if OUT.exists() else None
    src = sources()
    deps = src + [p for p in (HERE / "mini").rglob("*") if p.is_file()] + [p for p in (HERE / "ceres_cfg").rglob("*") if p.is_file()]
    if not force and OUT.exists() and all(OUT.stat().st_mtime >= d.stat().st_mtime for d in deps):
        return OUT
    objdir = OUTDIR / "ceres_obj"
    objdir.mkdir(parents=True, exist_ok=True)
    newest_hdr = max(d.stat().st_mtime for d in deps if d not in src)

    def compile_one(s):
        o = objdir / (s.parent.name + "_" + s.stem + ".o")
        if not force and o.exists() and o.stat().st_mtime >= max(s.stat().st_mtime, newest_hdr):
            return o, None
        r = subprocess.run(["g++", *FLAGS, *INC, "-c", str(s), "-o", str(o)], capture_output=True, text=True)
        return o, (r.stderr if r.returncode else None)

    with ThreadPoolExecutor(max_workers=min(16, os.cpu_count() or 4)) as ex:
        results = list(ex.map(compile_one, src))
    errs = [(o, e) for o, e in results if e]
    if errs:
        for o, e in errs[:5]:
            sys.stderr.write(f"--- {o.name}\n{e[:3000]}\n")
        raise RuntimeError(f"{len(errs)} Ceres sources failed to compile against the stand-in headers")
    cmd = ["g++", "-shared", "-o", str(OUT), *[str(o) for o, _ in results], "-lpthread", "-Wl,--no-undefined"]
    if verbose:
        print(" ".join(cmd[:4]), "...", flush=True)
    subprocess.check_call(cmd)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
