"""GPU tests of the large-window local-BA solve (csrc/ba_large.cu): ov2_localba_solve windows with more than 64 optimised
keyframes - the loop closer's looseBA and fullBA - against the C restatement of the oracle (oracle/ba_ref_c.c, mono) and the
numpy oracle (oracle/ba_ref.py, stereo), with the tolerances of test_localba_c5_size_150k_observations: same LM iteration
counts and termination, cost 1e-8 relative, poses and inverse depths 1e-6, outlier flags equal except threshold-borderline
observations.  Windows come from synth.make_loop_ba_problem: keyframes on a closed trajectory, so the reduced system is a
band plus the loop-closure blocks."""
import subprocess

import numpy as np
import pytest

from ov2slam_b200 import api, build, synth

pytestmark = pytest.mark.gpu

LOOSE = dict(max_iters_robust=5, max_iters_refine=0, function_tolerance=1e-4, apply_l2_after_robust=0)
FULL = dict(max_iters_robust=100, max_iters_refine=100, function_tolerance=1e-6)


def _clone(pb):
    return {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in pb.items()}


def _nopt(pb):
    return int((pb["pose_const"] == 0).sum())


def _oracle(pb, **opts):
    ref = _clone(pb)
    if pb.get("obs_type") is None:
        from oracle import ba_ref_c
        r = ba_ref_c.local_ba(ref, **opts)
    else:
        from oracle import ba_ref
        r = ba_ref.local_ba(ref, **opts)
    return ref, r


def _check(ctx, pb, **opts):
    ref, r = _oracle(pb, **opts)
    gpu = _clone(pb)
    g, flags = api.Optimizer(ctx).local_ba(gpu, **{k: int(v) if isinstance(v, bool) else v for k, v in opts.items()})
    assert (g["iters_robust"], g["iters_refine"]) == (r["iters_robust"], r["iters_refine"]), (g, r["iters_robust"], r["iters_refine"])
    assert g["termination"] == {"CONVERGENCE": 0, "NO_CONVERGENCE": 1, "FAILURE": 2}[r["termination"]]
    assert abs(g["final_cost"] - r["final_cost"]) <= 1e-8 * max(1.0, r["final_cost"])
    assert np.abs(gpu["pose"] - ref["pose"]).max() <= 1e-6
    assert np.abs(gpu["lm_invdepth"] - ref["lm_invdepth"]).max() <= 1e-6
    assert (flags != r["flags"]).sum() <= 4
    return g, gpu


@pytest.mark.parametrize("opts", [{}, LOOSE], ids=["localba", "looseba"])
def test_large_mono_loop_window_matches_oracle(ctx, opts):
    pb = synth.make_loop_ba_problem(1, 162, 8000)
    assert _nopt(pb) == 160
    g, _ = _check(ctx, pb, **opts)
    assert g["final_cost"] < g["initial_cost"]


@pytest.mark.parametrize("opts", [{}, LOOSE], ids=["localba", "looseba"])
def test_large_stereo_loop_window_matches_oracle(ctx, opts):
    pb = synth.make_loop_ba_problem(2, 121, 5000, stereo=True)
    assert _nopt(pb) == 120 and set(pb["obs_type"].tolist()) == {0, 1, 2}
    _check(ctx, pb, **opts)


def test_large_fullba_options_match_oracle(ctx):
    pb = synth.make_loop_ba_problem(3, 122, 6000)
    assert _nopt(pb) == 120
    g, _ = _check(ctx, pb, **FULL)
    assert g["iters_robust"] > 5


@pytest.mark.parametrize("nkf,kernel", [(66, "ba_lm_kernel"), (67, "ba_large_kernel")])
def test_capacity_boundary_64_and_65_optimised_keyframes(ctx, nkf, kernel):
    """64 optimised keyframes still run ba_lm_kernel; 65 run the large-window kernel; both equal the oracle."""
    pb = synth.make_loop_ba_problem(4, nkf, 4000)
    assert _nopt(pb) == nkf - 2
    ctx.profile(True)
    try:
        _check(ctx, pb)
        rep = ctx.profile_report()
    finally:
        ctx.profile(False)
    assert kernel in rep, rep
    other = "ba_large_kernel" if kernel == "ba_lm_kernel" else "ba_lm_kernel"
    assert other not in rep, rep


def _permute_keyframes(pb, seed):
    """The same window with its keyframes in a random order (as a newest-first or hash-ordered window hands them over): the
    system's tile rows are then long and the fill far from a band."""
    rng = np.random.default_rng(seed)
    ncam = len(pb["pose"])
    perm = rng.permutation(ncam)                       # old index -> new index
    out = _clone(pb)
    inv = np.argsort(perm)
    for k in ("pose", "pose_const", "truth_pose"):
        out[k] = np.ascontiguousarray(pb[k][inv])
    out["lm_anchor_cam"] = perm[pb["lm_anchor_cam"]].astype(np.int32)
    out["obs_cam"] = perm[pb["obs_cam"]].astype(np.int32)
    return out


@pytest.mark.parametrize("ctas", ["1", "3", "40", None])
def test_large_group_sizes_and_permuted_keyframes(ctx, monkeypatch, ctas):
    """1, 3 and 40 CTAs and the kernel's own choice: with few CTAs every CTA takes several items of a block step (panel tiles,
    column tiles) and every warp several tile pairs of the trailing update.  A loop window in trajectory order and the same
    window with its keyframes shuffled (long tile rows), both against the oracle."""
    if ctas is None:
        monkeypatch.delenv("OV2_BA_CTAS", raising=False)
    else:
        monkeypatch.setenv("OV2_BA_CTAS", ctas)
    pb = synth.make_loop_ba_problem(12, 98, 4000)
    _check(ctx, pb)
    pp = _permute_keyframes(pb, 13)
    assert _nopt(pp) == 96
    _check(ctx, pp, **LOOSE)


def test_more_than_256_keyframes_in_total(ctx):
    """80 optimised keyframes plus 200 constant observer keyframes: 282 in the window (the small-window path stops at 256)."""
    pb = synth.make_loop_ba_problem(5, 82, 5000, nconst_extra=200)
    assert len(pb["pose"]) > 256 and _nopt(pb) == 80
    _check(ctx, pb)


def test_capacity_edge_1024_optimised_keyframes_noise_free(ctx):
    """1026 keyframes (1024 optimised), 1.2 M residual blocks, no noise, no outliers: poses recover the truth, the cost falls
    and the solve converges.  No oracle at this size: the CPU restatement's dense solve would take hours."""
    pb = synth.make_loop_ba_problem(6, api.OV2_BA_MAX_OPT_KEYFRAMES + 2, 200000, obs_per_pt=6, px_noise=0.0, outlier_frac=0.0)
    assert _nopt(pb) == api.OV2_BA_MAX_OPT_KEYFRAMES
    gpu = _clone(pb)
    g, flags = api.Optimizer(ctx).local_ba(gpu, max_iters_robust=30, function_tolerance=1e-12)
    assert g["final_cost"] < 1e-3 * g["initial_cost"]
    assert g["termination"] == 0
    assert np.abs(gpu["pose"][:, :3] - pb["truth_pose"][:, :3]).max() < 2e-3
    q = gpu["pose"][:, 3:] / np.linalg.norm(gpu["pose"][:, 3:], axis=1, keepdims=True)
    t = pb["truth_pose"][:, 3:]
    assert np.minimum(np.abs(q - t).max(1), np.abs(q + t).max(1)).max() < 2e-3      # rotations, up to the quaternion sign


def test_over_capacity_raises(ctx):
    pb = synth.make_loop_ba_problem(7, api.OV2_BA_MAX_OPT_KEYFRAMES + 3, 20000)
    assert _nopt(pb) == api.OV2_BA_MAX_OPT_KEYFRAMES + 1
    with pytest.raises(api.Ov2Error, match="CAPACITY"):
        api.Optimizer(ctx).local_ba(_clone(pb))


def test_device_resident_window_equals_host_window(ctx):
    import torch
    pb = synth.make_loop_ba_problem(8, 102, 6000)
    host = _clone(pb)
    rh, fh = api.Optimizer(ctx).local_ba(host)
    dev = {k: (torch.from_numpy(v.copy()).cuda() if isinstance(v, np.ndarray) and k not in ("truth_pose", "truth_invdepth") else v)
           for k, v in pb.items()}
    keys = ("K", "pose", "pose_const", "lm_anchor_cam", "lm_anchor_px", "lm_invdepth", "obs_cam", "obs_lm", "obs_px")
    p = api.BaProblem(len(pb["pose"]), len(pb["lm_invdepth"]), len(pb["obs_cam"]), *[dev[k].data_ptr() for k in keys], None, None, None)
    bo = api.BaOpts(**api.DEFAULT_BA_OPTS)
    res = api.BaResult()
    flags = torch.zeros(len(pb["obs_cam"]), dtype=torch.uint8, device="cuda")
    ctx.check(ctx.lib.ov2_localba_solve(ctx.h, api.C.byref(p), api.C.byref(bo), api.C.byref(res), flags.data_ptr()))
    torch.cuda.synchronize()
    # (the fp64 reductions into the reduced system run in no fixed order: equal up to summation order, as two host solves are)
    assert (res.iters_robust, res.iters_refine, res.termination) == (rh["iters_robust"], rh["iters_refine"], rh["termination"])
    assert abs(res.final_cost - rh["final_cost"]) <= 1e-9 * max(1.0, rh["final_cost"])
    assert np.abs(dev["pose"].cpu().numpy() - host["pose"]).max() <= 1e-8
    assert np.abs(dev["lm_invdepth"].cpu().numpy() - host["lm_invdepth"]).max() <= 1e-8
    assert (flags.cpu().numpy() != fh).sum() <= 2


def test_large_stop_request_skips_the_refinement(ctx):
    pb = synth.make_loop_ba_problem(9, 100, 5000)
    r0, _ = api.Optimizer(ctx).local_ba(_clone(pb))
    assert r0["iters_refine"] > 0
    api.request_stop_local_ba(ctx, True)
    try:
        b = _clone(pb)
        r1, _ = api.Optimizer(ctx).local_ba(b)
    finally:
        api.request_stop_local_ba(ctx, False)
    assert r1["iters_refine"] == 0 and r1["iters_robust"] == r0["iters_robust"] and r1["n_outliers_first"] == r0["n_outliers_first"]
    ref, _ = _oracle(pb, apply_l2_after_robust=False)
    assert np.abs(b["pose"] - ref["pose"]).max() <= 1e-6
    r2, _ = api.Optimizer(ctx).local_ba(_clone(pb))
    assert r2["iters_refine"] == r0["iters_refine"]


def _write_window(path, pb):
    import struct
    stereo = pb.get("obs_type") is not None
    ncam, npts, nobs = len(pb["pose"]), len(pb["lm_invdepth"]), len(pb["obs_cam"])
    with open(path, "wb") as f:
        f.write(struct.pack("4i", ncam, npts, nobs, int(stereo)))
        f.write(np.asarray(pb["K"], np.float64).tobytes())
        f.write(np.asarray(pb["Kr"] if stereo else pb["K"], np.float64).tobytes())
        f.write(np.asarray(pb["Trl"] if stereo else [0, 0, 0, 0, 0, 0, 1], np.float64).tobytes())
        for k, dt in (("pose", np.float64), ("pose_const", np.uint8), ("lm_anchor_cam", np.int32), ("lm_anchor_px", np.float64),
                      ("lm_invdepth", np.float64), ("obs_cam", np.int32), ("obs_lm", np.int32), ("obs_px", np.float64)):
            f.write(np.ascontiguousarray(pb[k], dt).tobytes())
        f.write(np.ascontiguousarray(pb["obs_type"] if stereo else np.zeros(nobs), np.uint8).tobytes())


@pytest.mark.parametrize("mode,stereo", [("loose", False), ("loose", True), ("full", False), ("full", True)])
def test_dropin_loose_and_full_ba_optimise_the_whole_range(ctx, tmp_path, mode, stereo):
    """The drop-in Optimizer::looseBA / fullBA on a synthetic map of 150 keyframes: every keyframe of the range but the gauge
    (2 mono / 1 stereo) is optimised - none held constant for capacity - and the map left behind equals the flat solve."""
    exe = build.build_optimizer_shim()
    pb = synth.make_loop_ba_problem(10 + stereo, 150, 4000, stereo=stereo)
    _write_window(tmp_path / "w.bin", pb)
    out = subprocess.run([str(exe), str(tmp_path / "w.bin"), str(tmp_path / "r.bin"), mode], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "held constant" not in out.stderr
    ncam, npts = len(pb["pose"]), len(pb["lm_invdepth"])
    raw = np.fromfile(tmp_path / "r.bin", np.uint8)
    pose = raw[:ncam * 56].view(np.float64).reshape(ncam, 7)
    invd = raw[ncam * 56:ncam * 56 + npts * 8].view(np.float64)
    ref = _clone(pb)
    if mode == "loose":
        res, _ = api.Optimizer(ctx).local_ba(ref, **LOOSE)
    else:
        res, _ = api.Optimizer(ctx).local_ba(ref, **FULL)
    assert res["final_cost"] < res["initial_cost"]
    moved = np.abs(pose[:, :3] - pb["pose"][:, :3]).max(1) > 0
    assert moved.sum() == ncam - (1 if stereo else 2)
    for c in range(ncam):
        assert np.abs(pose[c, :3] - ref["pose"][c, :3]).max() <= 1e-7
        q, r = pose[c, 3:], ref["pose"][c, 3:] / np.linalg.norm(ref["pose"][c, 3:])
        assert min(np.abs(q - r).max(), np.abs(q + r).max()) <= 1e-7
    alive = invd >= 0
    assert alive.mean() > 0.9
    assert np.abs(invd[alive] - ref["lm_invdepth"][alive]).max() <= 1e-6 * np.abs(ref["lm_invdepth"][alive]).max() + 1e-7
