"""Large-window local BA on one GPU (csrc/ba_large.cu): a loop-closure looseBA window (~300 optimised keyframes) and a
fullBA-sized window (~1000 optimised keyframes, ~1.5 M residual blocks) from synth.make_loop_ba_problem.

For each window: solve time (host clock around the call, which ends in a stream synchronise; after one warm-up solve) and the
kernel time from the context's event profile, LM iterations, the per-phase trace (OV2_BA_TRACE=1, a separate solve), the
factored tiles of the reduced system against the dense count, and the FP64 rate the blocked factorisation reached (its flops
from the tile pattern over the trace's factorisation time).  CPU arm on the 300-keyframe window only: oracle/ba_ref_c.c, a
single-threaded C restatement of the solve with a DENSE Cholesky of the reduced system - not Ceres' SPARSE_SCHUR.
GPU name, power limit and clocks are read in the same run.

    python scripts/bench_ba_large.py [--out profiles/ba_large_b200.json] [--no-cpu]
"""
from __future__ import annotations

import argparse
import json
import os
import re
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

from ov2slam_b200 import api, synth  # noqa: E402

LOOSE = dict(max_iters_robust=5, max_iters_refine=0, function_tolerance=1e-4, apply_l2_after_robust=0)
FULL = dict(max_iters_robust=100, max_iters_refine=100, function_tolerance=1e-6)
WINDOWS = {
    "looseba_300kf": dict(args=(21, 302, 30000), kw=dict(obs_per_pt=6), opts=LOOSE),
    "fullba_1000kf": dict(args=(22, 1002, 250000), kw=dict(obs_per_pt=6), opts=FULL),
}
TB = 32


def _clone(pb):
    return {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in pb.items()}


def tile_pattern(pb):
    """Fill tiles of the reduced system (the host planning of ba_large.cu, restated): keyframe blocks per landmark, closed
    under the symbolic factorisation."""
    const = pb["pose_const"].astype(bool)
    ncam = len(const)
    typ = pb.get("obs_type")
    real = np.ones(len(pb["obs_cam"]), bool) if typ is None else typ != 2
    used = np.zeros(ncam, bool)
    used[pb["obs_cam"][real]] = True
    used[pb["lm_anchor_cam"][pb["obs_lm"][real]]] = True
    lay = -np.ones(ncam, np.int64)
    sel = used & ~const
    lay[sel] = np.arange(sel.sum())
    nt = max(1, -(-6 * int(sel.sum()) // TB))
    T = np.zeros((nt, nt), bool)
    obs_l, obs_c = pb["obs_lm"][real], pb["obs_cam"][real]
    slots = {}
    for l, c in zip(obs_l.tolist(), obs_c.tolist()):
        slots.setdefault(l, {int(lay[pb["lm_anchor_cam"][l]])}).add(int(lay[c]))
    for s in slots.values():
        s = sorted(v for v in s if v >= 0)
        tr = sorted({t for v in s for t in (6 * v // TB, (6 * v + 5) // TB)})
        for i in tr:
            for j in tr:
                if i <= j:
                    T[i, j] = True
    np.fill_diagonal(T, True)
    for k in range(nt):
        j = k + 1 + np.nonzero(T[k, k + 1:])[0]
        if len(j) > 1:
            T[np.ix_(j, j)] = True
    return np.triu(T)


def factor_flops(T):
    """FP64 flops of one blocked factorisation over the fill tiles (diagonal Cholesky, panel solves, trailing updates)."""
    f = 0.0
    for k in range(len(T)):
        m = int(T[k, k + 1:].sum())
        f += TB ** 3 / 3 + m * TB ** 3 + (m * (m - 1) / 2) * 2 * TB ** 3 + m * TB ** 3   # off-diagonal pairs + diagonal pairs
    return f


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm,clocks.mem", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        return q
    except Exception as e:  # noqa: BLE001
        return f"unavailable: {e}"


def trace_run(name):
    """One solve of window `name` with OV2_BA_TRACE=1 in a child process; returns the parsed trace line."""
    env = dict(os.environ, OV2_BA_TRACE="1")
    out = subprocess.run([sys.executable, __file__, "--trace-child", name], capture_output=True, text=True, env=env, timeout=3600)
    line = next((ln for ln in out.stderr.splitlines() if ln.startswith("[ba trace]")), "")
    phases = {k: float(v) for k, v in re.findall(r" ([A-Za-z0-9:|]+) ([0-9.]+)us", line)}
    m = re.search(r"tiles=(\d+)/(\d+)", line)
    return dict(line=line, phases_us=phases, tiles=[int(m.group(1)), int(m.group(2))] if m else None, child_rc=out.returncode)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=str(ROOT / "profiles" / "ba_large_b200.json"))
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--trace-child", default=None)
    a = ap.parse_args()
    ctx = api.Context()
    if a.trace_child:
        w = WINDOWS[a.trace_child]
        pb = synth.make_loop_ba_problem(*w["args"], **w["kw"])
        api.Optimizer(ctx).local_ba(_clone(pb), **w["opts"])
        return
    res = {"gpu": gpu_info(), "windows": {}}
    for name, w in WINDOWS.items():
        pb = synth.make_loop_ba_problem(*w["args"], **w["kw"])
        T = tile_pattern(pb)
        nt = len(T)
        opt = api.Optimizer(ctx)
        opt.local_ba(_clone(pb), **w["opts"])                     # warm-up (module load, scratch growth)
        times, kms = [], []
        for _ in range(3):
            ctx.profile(True)
            x = _clone(pb)
            t0 = time.perf_counter()
            r, _ = opt.local_ba(x, **w["opts"])
            times.append(time.perf_counter() - t0)
            kms.append(ctx.profile_report().get("ba_large_kernel", (float("nan"), 0))[0])
            ctx.profile(False)
        tr = trace_run(name)
        iters = r["iters_robust"] + r["iters_refine"]
        ph = tr["phases_us"]
        chol_s = (ph.get("chol:panel", 0) + ph.get("chol:bar", 0) + ph.get("chol:update", 0)) * 1e-6
        flops = factor_flops(T)
        entry = dict(
            keyframes=len(pb["pose"]), optimised=int((pb["pose_const"] == 0).sum()), landmarks=len(pb["lm_invdepth"]),
            residual_blocks=len(pb["obs_cam"]), options=w["opts"], n=6 * int((pb["pose_const"] == 0).sum()),
            solve_s=times, solve_s_median=float(np.median(times)), kernel_ms=kms,
            iters_robust=r["iters_robust"], iters_refine=r["iters_refine"], termination=r["termination"],
            initial_cost=r["initial_cost"], final_cost=r["final_cost"],
            factored_tiles=int(T.sum()), dense_tiles=nt * (nt + 1) // 2, tiles_from_trace=tr["tiles"],
            factorisation_flops=flops, factorisation_s_per_solve=chol_s / max(iters, 1) if chol_s else None,
            factorisation_fp64_tflops=(flops * iters / chol_s / 1e12) if chol_s else None,
            trace=tr["line"])
        print(name, json.dumps({k: v for k, v in entry.items() if k != "trace"}), flush=True)
        if name == "looseba_300kf" and not a.no_cpu:
            from oracle import ba_ref_c
            ref = _clone(pb)
            t0 = time.perf_counter()
            rc = ba_ref_c.local_ba(ref, **w["opts"])
            entry["cpu_c_restatement_dense_cholesky_s"] = time.perf_counter() - t0
            entry["cpu_iters"] = [rc["iters_robust"], rc["iters_refine"]]
            entry["cpu_final_cost"] = rc["final_cost"]
            print("  cpu (C restatement with a dense Cholesky, 1 thread):", entry["cpu_c_restatement_dense_cholesky_s"], "s", flush=True)
        res["windows"][name] = entry
    res["gpu_after"] = gpu_info()
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    Path(a.out).write_text(json.dumps(res, indent=1))
    print(json.dumps({"gpu": res["gpu"]}))


if __name__ == "__main__":
    main()
