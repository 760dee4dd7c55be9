"""oracle/ba_ref.py::local_ba against the REAL Ceres 2.0: oracle/_ref/libov2ref_ceres.so is the Ceres vendored in the reference tree
(Thirdparty/ceres-solver/internal/ceres/*.cc: Problem, Program reduction, ResidualBlock + Corrector + HuberLoss, ProgramEvaluator,
TrustRegionMinimizer, LevenbergMarquardtStrategy, SchurEliminator, DENSE_SCHUR solver ...) compiled where it lies together with the
reference's own cost functions (src/ceres_parametrization.cpp) and a driver that sets the window up and runs the two-stage flow with
the Ceres calls Optimizer::localBA makes (oracle/ref_build/ceres_ba_ref.cpp).  Stand-ins: the linear-algebra header (this container
has no Eigen; oracle/ref_build/mini), Ceres' generated config.h, and aborting stubs for three files off the DENSE_SCHUR + LM path.
Every iteration Ceres records (cost, cost change, step norm, relative decrease, radius, gradient max-norm, accepted / rejected), the
termination, the outlier flags of both scans and the final state must equal the restatement's."""
import ctypes as C

import numpy as np
import pytest

from oracle import ba_ref as B
from oracle.ref_build import build_ceres_ref
from ov2slam_b200 import synth
from reference_calls import library

D, I, U = C.POINTER(C.c_double), C.POINTER(C.c_int32), C.POINTER(C.c_uint8)
TERM = {0: "CONVERGENCE", 1: "NO_CONVERGENCE", 2: "FAILURE"}


@pytest.fixture(scope="module")
def lib():
    def load():
        so = build_ceres_ref.build()
        return None if so is None else C.CDLL(str(so))
    with library("ceres", load) as lib:
        lib.ov2ref_local_ba.restype = C.c_int
        yield lib


def run_ceres(lib, pb, max_iters_robust=5, max_iters_refine=10, th=5.9915, ftol=1e-3, robust=1, l2=1, maxlog=128):
    pose = np.ascontiguousarray(pb["pose"], np.float64).copy()
    invd = np.ascontiguousarray(pb["lm_invdepth"], np.float64).copy()
    nobs = len(pb["obs_cam"])
    flags, summ, log, nlog = np.zeros(nobs, np.uint8), np.zeros((2, 8)), np.zeros((2, maxlog, 9)), np.zeros(2, np.int32)
    a = {k: np.ascontiguousarray(pb[k], t) for k, t in (("K", np.float64), ("pose_const", np.uint8), ("lm_anchor_cam", np.int32),
                                                        ("lm_anchor_px", np.float64), ("obs_cam", np.int32), ("obs_lm", np.int32), ("obs_px", np.float64))}
    st = pb.get("obs_type") is not None
    kr = np.ascontiguousarray(pb["Kr"], np.float64) if st else None
    trl = np.ascontiguousarray(pb["Trl"], np.float64) if st else None
    ty = np.ascontiguousarray(pb["obs_type"], np.uint8) if st else None
    n = lib.ov2ref_local_ba(len(pose), len(invd), nobs, a["K"].ctypes.data_as(D), kr.ctypes.data_as(D) if st else None,
                            trl.ctypes.data_as(D) if st else None, pose.ctypes.data_as(D), a["pose_const"].ctypes.data_as(U),
                            a["lm_anchor_cam"].ctypes.data_as(I), a["lm_anchor_px"].ctypes.data_as(D), invd.ctypes.data_as(D),
                            a["obs_cam"].ctypes.data_as(I), a["obs_lm"].ctypes.data_as(I), a["obs_px"].ctypes.data_as(D),
                            ty.ctypes.data_as(U) if st else None, max_iters_robust, max_iters_refine, C.c_double(th), C.c_double(ftol), robust, l2,
                            flags.ctypes.data_as(U), summ.ctypes.data_as(D), log.ctypes.data_as(D), maxlog, nlog.ctypes.data_as(I))
    return dict(solves=n, pose=pose, invd=invd, flags=flags, summ=summ, log=[log[k, :nlog[k]] for k in range(2)])


def rel(a, b, tol=1e-9):
    return abs(a - b) <= tol * max(abs(a), abs(b), 1e-30) + 1e-12


def compare_solve(rows, summ, entries, osum, tol=1e-9):
    """rows: Ceres' IterationSummary list of one Solve; entries: the restatement's log of the same solve."""
    ctl = {e["it"]: e for e in entries if e.get("ctl")}
    its = {e["it"]: e for e in entries if not e.get("ctl")}
    assert rel(summ[0], osum["initial_cost"]) and rel(summ[1], osum["final_cost"], tol) and TERM[int(summ[2])] == osum["termination"]
    assert rows[0][0] == 0 and rel(rows[0][3], osum["initial_cost"]) and rows[0][8] == 1e4
    nrej = 0
    for row in rows[1:]:
        k = int(row[0])
        e, c = its[k], ctl[k]
        assert row[1] == 1.0                                      # step valid
        ok = e["rho"] > 1e-3
        nrej += not ok
        assert bool(row[2]) == ok
        assert rel(row[3], e["cand_cost"], tol)                   # Ceres records the candidate's cost for rejected steps too
        # a cost change is a difference of two costs: its error scales with the costs (compared at 1e-9 of them), and so does the ratio's
        cc_tol = tol * max(e["x_cost"], e["cand_cost"])
        assert abs(row[4] - (e["x_cost"] - e["cand_cost"])) <= cc_tol + 1e-12
        assert abs(row[7] - e["rho"]) <= cc_tol / abs(e["mcc"]) + tol * abs(e["rho"])
        assert rel(row[6], np.sqrt(c["step2"]), tol)
        if k + 1 in its:
            assert rel(row[8], its[k + 1]["radius"], 10 * tol)           # radius after this iteration = the next one's
        if k + 1 in ctl:
            # gradient entries are sums of cancelling terms J^T r: compared at 1e-9 of the initial gradient's scale
            assert abs(row[5] - ctl[k + 1]["gmax"]) <= tol * max(rows[0][5], 1.0) + tol * abs(row[5])
    # the restatement counts the iteration in which a tolerance fired; Ceres returns before recording it
    assert osum["iterations"] in (int(rows[-1][0]), int(rows[-1][0]) + 1)
    return nrej


def check(lib, pb, tol=1e-9, **kw):
    ref = run_ceres(lib, pb, **{dict(max_iters_robust="max_iters_robust", max_iters_refine="max_iters_refine", robust="robust", l2="l2", th="th", ftol="ftol")[k]: v
                                for k, v in kw.items()})
    o = {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in pb.items()}
    log = []
    res = B.local_ba(o, max_iters_robust=kw.get("max_iters_robust", 5), max_iters_refine=kw.get("max_iters_refine", 10), huber_th=kw.get("th", 5.9915),
                     function_tolerance=kw.get("ftol", 1e-3), use_robust=bool(kw.get("robust", 1)), apply_l2_after_robust=bool(kw.get("l2", 1)), log=log)
    assert ref["solves"] == len(res["summaries"])
    # split the restatement's log per solve: `it` restarts at 1
    cuts = [i for i, e in enumerate(log) if e["it"] == 1 and (i == 0 or log[i - 1]["it"] != 1)]
    parts = [log[cuts[0]:cuts[1]], log[cuts[1]:]] if len(cuts) > 1 else [log]
    nrej = 0
    for s in range(ref["solves"]):
        nrej += compare_solve(ref["log"][s], ref["summ"][s], parts[s], res["summaries"][s], tol)
    assert np.array_equal(ref["flags"], res["flags"])
    assert np.abs(ref["pose"] - o["pose"]).max() <= tol and np.abs(ref["invd"] - o["lm_invdepth"]).max() <= tol
    return res, nrej


@pytest.mark.parametrize("seed,ncam,npts,nobs", [(3, 6, 200, 800), (5, 8, 400, 1600), (11, 5, 120, 400)])
def test_mono_two_stage_solve_equals_real_ceres(lib, seed, ncam, npts, nobs):
    res, _ = check(lib, synth.make_ba_problem(seed, ncam, npts, nobs))
    assert res["n_outliers_first"] > 0 and res["iters_refine"] > 0      # both stages ran (Huber kept in the refinement: mono window)


def test_stereo_window_equals_real_ceres(lib):
    res, _ = check(lib, synth.make_ba_problem(21, 6, 200, 800, stereo=True))
    assert res["n_outliers_first"] > 0 and res["iters_refine"] > 0      # refinement with the trivial loss (left and right lists non-empty)


def test_c3_size_window_equals_real_ceres(lib):
    check(lib, synth.make_ba_problem(0, 10, 2000, 8000))


def test_options_trivial_loss_and_single_stage(lib):
    pb = synth.make_ba_problem(7, 6, 200, 800)
    check(lib, pb, robust=0)
    check(lib, pb, l2=0)
    check(lib, pb, max_iters_robust=2, max_iters_refine=3)                # NO_CONVERGENCE at the iteration cap
    check(lib, pb, ftol=1e-9, max_iters_robust=30, max_iters_refine=30)
    # the budgets of Optimizer::looseBA (optimizer.cpp:1298-1299: one 5-iteration solve at 1e-4) and fullBA (:2056: 100 iterations at Ceres'
    # default 1e-6), which the drop-ins pass to the same solve
    check(lib, pb, ftol=1e-4, max_iters_robust=5, l2=0)
    check(lib, pb, ftol=1e-6, max_iters_robust=100, max_iters_refine=100)


def test_rejected_steps_follow_real_ceres(lib):
    """Windows whose first steps overshoot (inverse depths off by e^+-1.5, poses by 0.3 m): Ceres rejects steps, shrinks the radius
    (/2, /4, ...) and reuses the diagonal.  These trajectories are ill-conditioned (points pass through cameras, costs of 1e5), so
    rounding differences grow from iteration to iteration: same decisions, values compared at 1e-5."""
    nrej = 0
    for seed in (40, 42, 43, 44):
        pb = synth.make_ba_problem(seed, 6, 150, 600)
        rng = np.random.default_rng(seed)
        pb["lm_invdepth"] = pb["lm_invdepth"] * np.exp(rng.normal(0, 1.5, len(pb["lm_invdepth"])))
        pb["pose"][2:, :3] += rng.normal(0, 0.3, pb["pose"][2:, :3].shape)
        nrej += check(lib, pb, tol=1e-5, max_iters_robust=12, max_iters_refine=12)[1]
    assert nrej >= 10


def test_bal_structure_window_equals_real_ceres(lib):
    """The observation graph of Ceres' own bundle-adjustment test problem (problem-16-22106-pre.txt, tests/ba_fixture.py): a 2 000-landmark
    subset with track lengths 2 .. 14 and an uneven covisibility pattern (16 keyframes, 14 optimised: a 84 x 84 reduced system)."""
    import sys
    from pathlib import Path
    sys.path.insert(0, str(Path(__file__).parent))
    import ba_fixture as F
    pb = F.bal_window(seed=1, max_pts=2000)
    pb = {k: v for k, v in pb.items() if k != "truth_pose"}
    res, _ = check(lib, pb)
    assert res["n_outliers_first"] > 0


@pytest.mark.parametrize("seed,npts,noise,nout", [(1, 300, 0.5, 30), (2, 120, 1.0, 0), (3, 700, 0.3, 100), (4, 40, 0.5, 8)])
def test_ceres_pnp_equals_real_ceres(lib, seed, npts, noise, nout):
    """oracle/pnp_ref.py::ceres_pnp against MultiViewGeometry::ceresPnP's Ceres calls (multi_view_geometry.cpp:492-588: one pose block,
    ReprojectionErrorSE3 with sigma = 2^octave behind a Huber wrapper, DENSE_QR, 5 iterations, outlier scan, L2 refinement on the inliers)
    run by the real Ceres on the reference's cost function: same outliers, same verdict, same pose."""
    from oracle import pnp_ref as P
    rng = np.random.default_rng(seed)
    K = np.array([458.654, 457.296, 367.215, 248.375], np.float32).astype(np.float64)      # the reference passes floats
    q = B.quat_normalize(np.array([0.05, -0.02, 0.03, 1.0]) + rng.normal(0, 0.1, 4))
    Ttrue = np.concatenate([rng.normal(0, 0.5, 3), q])
    R, t = B.quat_to_rot(q), Ttrue[:3]
    pc = np.stack([rng.uniform(-2, 2, npts), rng.uniform(-1.5, 1.5, npts), rng.uniform(2, 9, npts)], 1)
    w = pc @ R.T + t
    px = np.stack([K[0] * pc[:, 0] / pc[:, 2] + K[2], K[1] * pc[:, 1] / pc[:, 2] + K[3]], 1) + rng.normal(0, noise, (npts, 2))
    px[:nout] += rng.uniform(8, 40, (nout, 2)) * rng.choice([-1, 1], (nout, 2))
    scales = rng.integers(0, 3, npts).astype(np.int32)
    T0 = Ttrue.copy()
    T0[:3] += rng.normal(0, 0.05, 3)
    T0[3:] = B.quat_normalize(T0[3:] + rng.normal(0, 0.01, 4))
    for robust, l2 in ((1, 1), (1, 0), (0, 0)):
        T = T0.copy()
        out, summ = np.zeros(npts, np.uint8), np.zeros((2, 8))
        lib.ov2ref_ceres_pnp.restype = C.c_int
        rc = lib.ov2ref_ceres_pnp(npts, np.ascontiguousarray(px).ctypes.data_as(D), np.ascontiguousarray(w).ctypes.data_as(D), scales.ctypes.data_as(I),
                                  T.ctypes.data_as(D), 5, C.c_double(5.9915), robust, l2, K.ctypes.data_as(D), out.ctypes.data_as(U), summ.ctypes.data_as(D))
        ok, pose, outliers = P.ceres_pnp(px, w, T0.copy(), K, nmaxiter=5, chi2th=5.9915, use_robust=bool(robust), apply_l2_after_robust=bool(l2), scales=scales)
        assert rc in (0, 1) and bool(rc) == ok
        assert np.array_equal(np.nonzero(out)[0], outliers) and (nout == 0 or len(outliers) >= nout // 2)
        assert np.abs(T - pose).max() <= 1e-9


def test_c_restatement_used_as_cpu_baseline_equals_real_ceres(lib):
    """oracle/ba_ref_c.c (what bench.py times as the single-thread CPU baseline of the localBA legs) against the real Ceres directly:
    same outlier flags, final cost and state on a C3-size window and a smaller one (the C restatement is mono only, as the bench legs are).  (The real-Ceres build itself is
    not used for timing: on the stand-in linear algebra it runs 13 solves/s on C3 where the C restatement runs ~110 - the restatement
    is the faster, i.e. the more conservative, baseline.)"""
    from oracle import ba_ref_c
    for pb in (synth.make_ba_problem(0, 10, 2000, 8000), synth.make_ba_problem(23, 7, 300, 1200)):
        ref = run_ceres(lib, pb)
        o = {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in pb.items()}
        rc = ba_ref_c.local_ba(o)
        assert np.array_equal(ref["flags"], rc["flags"])
        last = ref["summ"][ref["solves"] - 1]
        assert abs(last[1] - rc["final_cost"]) <= 1e-9 * rc["final_cost"]
        assert np.abs(ref["pose"] - o["pose"]).max() <= 1e-9 and np.abs(ref["invd"] - o["lm_invdepth"]).max() <= 1e-9


def test_product_pnp_solver_code_equals_real_ceres(lib, tmp_path):
    """The PRODUCT's ceresPnP solve (ov2slam_b200/csrc/pnp_math.cuh - the code the CUDA kernel instantiates - compiled for the host with
    its single-lane context) directly against the real Ceres running the reference's cost function: same verdict, same rejected blocks,
    pose to 1e-9 (normal equations in the kernel code, DENSE_QR in Ceres)."""
    import subprocess
    from pathlib import Path
    root = Path(__file__).resolve().parents[1]
    src = tmp_path / "p.cpp"
    src.write_text(r"""
#include "%s/ov2slam_b200/csrc/pnp_math.cuh"
#include <vector>
extern "C" int pnp_host(int n, const double* unpx, const double* wpts, const int* scales, const double* K, double* pose, int nmaxiter, float chi2th,
                        int use_robust, int apply_l2, unsigned char* flags) {
    pnp::Problem P; P.n = n; P.unpx = unpx; P.wpts = wpts; P.scales = scales;
    for (int i = 0; i < 4; ++i) P.K[i] = K[i];
    std::vector<double> chi2(n); std::vector<unsigned char> dep(n), work(n);
    pnp::SerialPar par; pnp::Summary S;
    return pnp::ceres_pnp(par, P, pose, nmaxiter, chi2th, use_robust != 0, apply_l2 != 0, chi2.data(), dep.data(), flags, work.data(), S) ? 1 : 0;
}""" % root)
    so = tmp_path / "libp.so"
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fPIC", "-shared", "-o", str(so), str(src)])
    host = C.CDLL(str(so))
    lib.ov2ref_ceres_pnp.restype = C.c_int
    K = np.array([458.654, 457.296, 367.215, 248.375], np.float32).astype(np.float64)
    rng = np.random.default_rng(8)
    nbad_total = 0
    for case in range(10):
        n = int(rng.integers(40, 500))
        q = B.quat_normalize(np.array([0.0, 0.0, 0.0, 1.0]) + rng.normal(0, 0.15, 4))
        Ttrue = np.concatenate([rng.normal(0, 0.5, 3), q])
        pc = np.stack([rng.uniform(-2, 2, n), rng.uniform(-1.5, 1.5, n), rng.uniform(2, 10, n)], 1)
        w = np.ascontiguousarray(pc @ B.quat_to_rot(q).T + Ttrue[:3])
        px = np.stack([K[0] * pc[:, 0] / pc[:, 2] + K[2], K[1] * pc[:, 1] / pc[:, 2] + K[3]], 1) + rng.normal(0, 0.6, (n, 2))
        nbad = n // 8 if case % 2 else 0
        px[:nbad] += rng.uniform(15, 60, (nbad, 2))
        px = np.ascontiguousarray(px)
        scales = rng.integers(0, 3, n).astype(np.int32)
        T0 = B.pose_plus(Ttrue, np.concatenate([rng.normal(0, 0.05, 3), rng.normal(0, 0.02, 3)]))
        for l2 in (1, 0):
            Tc, Th = T0.copy(), T0.copy()
            oc, oh, summ = np.zeros(n, np.uint8), np.zeros(n, np.uint8), np.zeros((2, 8))
            rc = lib.ov2ref_ceres_pnp(n, px.ctypes.data_as(D), w.ctypes.data_as(D), scales.ctypes.data_as(I), Tc.ctypes.data_as(D), 5, C.c_double(5.9915),
                                      1, l2, K.ctypes.data_as(D), oc.ctypes.data_as(U), summ.ctypes.data_as(D))
            rh = host.pnp_host(n, px.ctypes.data_as(D), w.ctypes.data_as(D), scales.ctypes.data_as(I), K.ctypes.data_as(D), Th.ctypes.data_as(D), 5,
                               C.c_float(5.9915), 1, l2, oh.ctypes.data_as(U))
            assert rc in (0, 1) and rc == rh
            assert np.array_equal(oc, oh)
            assert np.abs(Tc - Th).max() <= 1e-9
            nbad_total += int(oc.sum())
    assert nbad_total > 100
