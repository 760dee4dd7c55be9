"""The REFERENCE'S OWN Optimizer::localBA run end to end (oracle/_ref/libov2ref_map.so: src/optimizer.cpp, frame.cpp, map_point.cpp,
map_manager.cpp, camera_calibration.cpp, multi_view_geometry.cpp compiled where they lie, with the Ceres 2.0 and Sophus of the reference
tree; stand-ins only for Eigen, the OpenCV containers and PCL) on maps built through the reference's own map API:
  * what it leaves in the map equals the flat solve (oracle/ba_ref.py::local_ba, == the GPU solve) of the same window, with the
    keyframes the reference itself chose to hold constant;
  * the drop-in Optimizer::localBA (ov2slam_b200/host/optimizer_localba_gpu.cpp), with its device call recorded instead of executed,
    hands the GPU the same window: the same constant keyframes (the reference's gauge walk over its keyframe hash map fixes ONE
    keyframe where the comment promises two), the same landmarks and observations."""
import ctypes as C
import os
import subprocess
from pathlib import Path

import numpy as np
import pytest

from oracle import ba_ref as B
from ov2slam_b200 import build, synth
from reference_calls import library

pytest.importorskip("cv2")
ROOT = Path(__file__).resolve().parents[1]
D, I, U = C.POINTER(C.c_double), C.POINTER(C.c_int32), C.POINTER(C.c_uint8)


@pytest.fixture(scope="module")
def lib():
    from oracle.ref_build import build_map_ref, cv_callbacks as CB

    def load():
        so = build_map_ref.build()
        if so is None:
            return None
        lib = C.CDLL(str(so))
        cb = CB._Callbacks(*[C.cast(f, C.c_void_p) for f in CB._KEEP])
        lib.ov2ref_cv_set_callbacks(C.byref(cb))
        return lib
    with library("map", load) as lib:
        lib.ov2ref_run_local_ba.restype = C.c_int
        yield lib


def reference_local_ba(lib, pb, nmin_covscore=25, mode=0):
    ncam, npts, nobs = len(pb["pose"]), len(pb["lm_invdepth"]), len(pb["obs_cam"])
    a = {k: np.ascontiguousarray(pb[k], t) for k, t in (("K", np.float64), ("pose", np.float64), ("lm_anchor_cam", np.int32), ("lm_anchor_px", np.float64),
                                                        ("lm_invdepth", np.float64), ("obs_cam", np.int32), ("obs_lm", np.int32), ("obs_px", np.float64))}
    pose, xyz, alive, left = np.zeros((ncam, 7)), np.zeros((npts, 3)), np.zeros(npts, np.uint8), np.zeros(npts, np.int32)
    rc = lib.ov2ref_run_local_ba(ncam, npts, nobs, a["K"].ctypes.data_as(D), 752, 480, a["pose"].ctypes.data_as(D), a["lm_anchor_cam"].ctypes.data_as(I),
                                 a["lm_anchor_px"].ctypes.data_as(D), a["lm_invdepth"].ctypes.data_as(D), a["obs_cam"].ctypes.data_as(I),
                                 a["obs_lm"].ctypes.data_as(I), a["obs_px"].ctypes.data_as(D), nmin_covscore, mode, pose.ctypes.data_as(D), xyz.ctypes.data_as(D),
                                 alive.ctypes.data_as(U), left.ctypes.data_as(I))
    assert rc == 0
    return pose, xyz, alive.astype(bool), left


def inside_image(pb, w=752, h=480, margin=2.0):
    """The window without the observations (and landmarks) whose pixels fall outside the image: the reference's Frame keeps its keypoints
    in a grid over the image and indexes it unchecked."""
    ok_l = (pb["lm_anchor_px"][:, 0] >= margin) & (pb["lm_anchor_px"][:, 0] < w - margin) & (pb["lm_anchor_px"][:, 1] >= margin) & (pb["lm_anchor_px"][:, 1] < h - margin)
    ok_o = (pb["obs_px"][:, 0] >= margin) & (pb["obs_px"][:, 0] < w - margin) & (pb["obs_px"][:, 1] >= margin) & (pb["obs_px"][:, 1] < h - margin)
    ok_o &= ok_l[pb["obs_lm"]]
    ok_l &= np.bincount(pb["obs_lm"][ok_o], minlength=len(ok_l)) > 0
    ok_o &= ok_l[pb["obs_lm"]]
    new_id = np.cumsum(ok_l) - 1
    out = dict(pb)
    for k in ("lm_anchor_cam", "lm_anchor_px", "lm_invdepth"):
        out[k] = pb[k][ok_l].copy()
    for k in ("obs_cam", "obs_px"):
        out[k] = pb[k][ok_o].copy()
    out["obs_lm"] = new_id[pb["obs_lm"][ok_o]].astype(np.int32)
    out["pose"] = pb["pose"].copy()
    return out


def world_points(pb, pose, invd):
    fx, fy, cx, cy = pb["K"]
    ua, ca = pb["lm_anchor_px"], pb["lm_anchor_cam"]
    bear = np.stack([(ua[:, 0] - cx) / fx, (ua[:, 1] - cy) / fy, np.ones(len(ua))], 1) / invd[:, None]
    R = B.quat_to_rot(B.quat_normalize(pose[ca, 3:]))
    return (R @ bear[..., None])[..., 0] + pose[ca, :3]


@pytest.mark.parametrize("seed,ncam,npts,nobs", [(3, 6, 200, 800), (12, 8, 300, 1300), (17, 5, 150, 520)])
def test_reference_local_ba_leaves_the_map_of_the_flat_solve(lib, seed, ncam, npts, nobs, capfd):
    pb = synth.make_ba_problem(seed, ncam, npts, nobs)
    pose, xyz, alive, left = reference_local_ba(lib, pb)
    const = np.abs(pose - pb["pose"]).max(1) <= 1e-14          # (a constant keyframe comes back re-normalised: equal to rounding)
    assert const[0] and const.sum() == 1                       # every keyframe covisible: only keyframe 0 ends up constant (see the module docstring)
    o = {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in pb.items()}
    o["pose_const"] = const.astype(np.uint8)
    res = B.local_ba(o)
    assert res["n_outliers_first"] > 0 and res["iters_refine"] > 0
    assert np.abs(pose - o["pose"]).max() <= 1e-9
    w = world_points(pb, o["pose"], o["lm_invdepth"])
    assert alive.mean() > 0.95 and np.abs(w[alive] - xyz[alive]).max() <= 1e-8
    # observations the two scans flagged are removed from the map (optimizer.cpp:741-897): per landmark, observers left = observers - flagged
    nobs_of = 1 + np.bincount(pb["obs_lm"], minlength=npts)
    bad_of = np.bincount(pb["obs_lm"], weights=(res["flags"] != 0).astype(float), minlength=npts).astype(int)
    assert np.array_equal(left[alive], (nobs_of - bad_of)[alive])


def _write_window(path, pb):
    ncam, npts, nobs = len(pb["pose"]), len(pb["lm_invdepth"]), len(pb["obs_cam"])
    with open(path, "wb") as f:
        f.write(np.array([ncam, npts, nobs, 0], np.int32).tobytes())
        f.write(np.asarray(pb["K"], np.float64).tobytes() + np.zeros(4).tobytes() + np.array([0, 0, 0, 0, 0, 0, 1.0]).tobytes())
        for k, t in (("pose", np.float64), ("pose_const", np.uint8), ("lm_anchor_cam", np.int32), ("lm_anchor_px", np.float64), ("lm_invdepth", np.float64),
                     ("obs_cam", np.int32), ("obs_lm", np.int32), ("obs_px", np.float64)):
            f.write(np.ascontiguousarray(pb[k], t).tobytes())
        f.write(np.zeros(nobs, np.uint8).tobytes())


@pytest.mark.parametrize("seed,ncam,npts,nobs", [(3, 6, 200, 800), (12, 8, 300, 1300)])
def test_drop_in_local_ba_hands_over_the_window_the_reference_solves(lib, tmp_path, seed, ncam, npts, nobs):
    pb = synth.make_ba_problem(seed, ncam, npts, nobs)
    pose, _, _, _ = reference_local_ba(lib, pb)
    ref_const = np.abs(pose - pb["pose"]).max(1) <= 1e-14
    exe = build.build_optimizer_shim()
    rec = tmp_path / "librec.so"
    subprocess.check_call(["gcc", "-shared", "-fPIC", "-O1", "-o", str(rec), str(ROOT / "tests" / "helpers" / "ba_dump.c")])
    _write_window(tmp_path / "w.bin", pb)
    env = dict(os.environ, LD_PRELOAD=str(rec), OV2_BA_DUMP=str(tmp_path / "d.bin"))
    out = subprocess.run([str(exe), str(tmp_path / "w.bin"), str(tmp_path / "r.bin"), "gauge"], capture_output=True, text=True, timeout=120, env=env)
    assert out.returncode == 0, out.stdout + out.stderr
    raw = np.fromfile(tmp_path / "d.bin", np.uint8)
    n = raw[:12].view(np.int32)
    dcam, dpts, dobs = int(n[0]), int(n[1]), int(n[2])
    dpose = raw[12:12 + 56 * dcam].view(np.float64).reshape(dcam, 7)
    dconst = raw[12 + 56 * dcam:12 + 57 * dcam].astype(bool)
    assert (dcam, dpts, dobs) == (ncam, npts, nobs)
    # keyframes by identity (their pose): the drop-in's constant set is the reference's
    for c in range(dcam):
        k = int(np.argmin(np.abs(pb["pose"] - dpose[c]).sum(1)))
        assert np.abs(pb["pose"][k] - dpose[c]).max() <= 1e-12 and dconst[c] == ref_const[k]


@pytest.mark.parametrize("mode,seed", [(1, 4), (2, 4), (1, 9), (2, 9)])
def test_reference_loose_and_full_ba_leave_the_map_of_the_flat_solve(lib, mode, seed):
    """Optimizer::looseBA (keyframe range, one 5-iteration solve at 1e-4, optimizer.cpp:900-1671) and fullBA (all keyframes, 100 + 100
    iterations at Ceres' default tolerance, :1674-2331), the reference's own code end to end: the first two keyframes of the range are held
    constant (mono) and the map they leave equals the flat solve with those budgets - what the drop-ins pass to the GPU solve
    (tests/test_host_shim.py::test_optimizer_loose_and_full_ba_shims)."""
    pb = inside_image(synth.make_ba_problem(seed, 6, 200, 800))
    pose, xyz, alive, _ = reference_local_ba(lib, pb, mode=mode)
    const = np.abs(pose - pb["pose"]).max(1) <= 1e-14
    assert list(np.nonzero(const)[0]) == [0, 1]
    o = {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in pb.items()}
    o["pose_const"] = const.astype(np.uint8)
    if mode == 1:
        B.local_ba(o, max_iters_robust=5, max_iters_refine=0, function_tolerance=1e-4, apply_l2_after_robust=False)
    else:
        B.local_ba(o, max_iters_robust=100, max_iters_refine=100, function_tolerance=1e-6)
    assert np.abs(pose - o["pose"]).max() <= 1e-8
    w = world_points(pb, o["pose"], o["lm_invdepth"])
    assert alive.mean() > 0.9 and np.abs(w[alive] - xyz[alive]).max() <= 1e-7


@pytest.mark.parametrize("seed,nkps,ncand", [(5, 500, 260), (6, 1200, 700), (7, 300, 400)])
def test_match_to_map_equals_the_reference_source(lib, seed, nkps, ncand):
    """The REFERENCE'S OWN Mapper::matchToMap (src/mapper.cpp:576-774, with Frame / MapManager / MapPoint of the reference) on a map built
    from a flattened matching scene (undistorted calibration): the pairs it returns are those of oracle/match_ref.py::match_to_map (which
    the GPU operator is compared with) for the same candidate order.  Poses pass through unit quaternions on the reference's side, so a
    projection may differ in the last bit: at most 1 % of the pairs may differ."""
    from oracle import match_ref as M
    sc = synth.make_match_scene(seed, nkps=nkps, ncand=ncand, nkfs=9, distorted=False)
    nmps, nkfs = len(sc["mp_xyz"]), len(sc["kf_Tcw"])
    a = {k: np.ascontiguousarray(sc[k], t) for k, t in (("K", np.float64), ("Tcw", np.float64), ("kf_Tcw", np.float64), ("mp_xyz", np.float64), ("kp_px", np.float32),
                                                        ("kp_lm", np.int32), ("mp_desc_ptr", np.int32), ("desc", np.uint8), ("mp_obs_ptr", np.int32),
                                                        ("obs_kf", np.int32), ("obs_px", np.float32), ("cand_mp", np.int32))}
    order, pairs = np.zeros(ncand, np.int32), np.zeros((nkps, 2), np.int32)
    F32 = C.POINTER(C.c_float)
    lib.ov2ref_match_to_map.restype = C.c_int
    n = lib.ov2ref_match_to_map(nkps, nmps, nkfs, ncand, a["K"].ctypes.data_as(D), sc["img_w"], sc["img_h"], sc["ncellsize"], a["Tcw"].ctypes.data_as(D),
                                a["kf_Tcw"].ctypes.data_as(D), a["mp_xyz"].ctypes.data_as(D), a["kp_px"].ctypes.data_as(F32), a["kp_lm"].ctypes.data_as(I),
                                a["mp_desc_ptr"].ctypes.data_as(I), a["desc"].ctypes.data_as(U), a["mp_obs_ptr"].ctypes.data_as(I), a["obs_kf"].ctypes.data_as(I),
                                a["obs_px"].ctypes.data_as(F32), a["cand_mp"].ctypes.data_as(I), C.c_float(2.0), C.c_float(0.2), order.ctypes.data_as(I),
                                pairs.ctypes.data_as(I))
    got = {(int(p[0]), int(p[1])) for p in pairs[:n]}
    ref = dict(sc, cand_mp=order)
    kp_match = M.match_to_map(ref)[2]
    want = {(int(sc["kp_lm"][j]), int(order[c])) for j, c in enumerate(kp_match) if c >= 0}
    assert len(want) > 40
    assert len(want ^ got) <= max(1, len(want) // 100)


@pytest.mark.parametrize("rect", [1, 0])
def test_stereo_matching_equals_the_reference_source(lib, rect):
    """The REFERENCE'S OWN MapManager::stereoMatching (src/map_manager.cpp:367-611, calling its own fbKltTracking / getLineMinSAD) on a synthetic
    stereo keyframe over a textured pair (16 px disparity), the arithmetic answered by the real library: the keypoints that become stereo
    keypoints and their right pixels are those of the flow restatement tests/test_host_shim.py checks the drop-in against
    (`_stereo_flow`), fed with the same library functions - so the drop-in's flow is the reference's."""
    import sys
    import cv2
    sys.path.insert(0, str(Path(__file__).parent))
    import test_host_shim as H
    from oracle import image_ref as R
    w, h, disp = 752, 480, 16.0
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float64)
    tex = lambda u: np.rint(128 + 50 * np.sin(0.11 * u + 0.07 * yy) + 40 * np.sin(0.05 * u - 0.13 * yy + 1) + 30 * np.sin(0.31 * u + 0.23 * yy + 2)).astype(np.uint8)
    left, right = tex(xx), tex(xx + disp)
    sc = H._stereo_scene(91 + rect, rect, nkps=260, depth=458.654 * 0.11 / disp)
    lv_l, lv_r = [left], [right]
    for _ in range(3):
        lv_l.append(cv2.pyrDown(lv_l[-1]))
        lv_r.append(cv2.pyrDown(lv_r[-1]))
    n = len(sc["lmid"])
    PP = C.POINTER(C.c_uint8) * 4
    pl, pr = PP(*[a.ctypes.data_as(U) for a in lv_l]), PP(*[a.ctypes.data_as(U) for a in lv_r])
    rows, cols = np.array([a.shape[0] for a in lv_l], np.int32), np.array([a.shape[1] for a in lv_l], np.int32)
    order, st, rpx = np.zeros(n, np.int32), np.zeros(n, np.int32), np.zeros((n, 2), np.float32)
    a = dict(K=np.ascontiguousarray(sc["K"], np.float64), rig=np.ascontiguousarray(np.concatenate([sc["trig"], H._quat_of(sc["Rrig"])]), np.float64),
             Twc=np.ascontiguousarray(np.concatenate([sc["twc"], H._quat_of(sc["Rwc"])]), np.float64), lmid=np.ascontiguousarray(sc["lmid"], np.int32),
             is3d=np.ascontiguousarray(sc["is3d"], np.int32), has=np.ascontiguousarray(sc["has_mp"], np.int32), px=np.ascontiguousarray(sc["px"], np.float32),
             wpt=np.ascontiguousarray(sc["wpt"], np.float64))
    lib.ov2ref_stereo_matching.restype = C.c_int
    m = lib.ov2ref_stereo_matching(n, rect, a["K"].ctypes.data_as(D), a["K"].ctypes.data_as(D), a["rig"].ctypes.data_as(D), a["Twc"].ctypes.data_as(D), w, h, 35,
                                   a["lmid"].ctypes.data_as(I), a["is3d"].ctypes.data_as(I), a["has"].ctypes.data_as(I), a["px"].ctypes.data_as(C.POINTER(C.c_float)),
                                   a["wpt"].ctypes.data_as(D), pl, pr, rows.ctypes.data_as(I), cols.ctypes.data_as(I), order.ctypes.data_as(I),
                                   st.ctypes.data_as(I), rpx.ctypes.data_as(C.POINTER(C.c_float)))
    assert m == n

    def klt(pts, pri, nlv):
        out, status = R._fb_klt(R._lk_cv2, left, right, pts, pri, 9, nlv, 30.0, 0.5, 30, R.KLT_EPS)
        return out, status.astype(bool)

    def sad(sp):
        subpix = lambda src, ws, cx, cy: cv2.getRectSubPix(src, (ws, ws), (float(cx), float(cy)))
        return np.array([R.line_min_sad_ref(lv_l[3], lv_r[3], (float(p[0]), float(p[1])), 7, True, subpix=subpix)[0] for p in sp], np.float32)

    _, want, _ = H._stereo_flow(sc, order, klt=klt, sad=sad)
    got = {int(l) for l, s in zip(order, st) if s}
    assert got == set(want) and len(got) > 0.6 * n
    for l, p in zip(order, rpx):
        if int(l) in want:
            assert np.abs(p - want[int(l)]).max() <= 1e-4


@pytest.mark.parametrize("detector,w,h,cs", [(0, 640, 480, 50), (1, 752, 480, 35)])
def test_extract_keypoints_equals_the_reference_source(lib, detector, w, h, cs):
    """The REFERENCE'S OWN MapManager::extractKeypoints (src/map_manager.cpp:286-341) - the caller of the detector and the descriptor that
    one front-end step mirrors (ov2_frontend_step / oracle frontend composite): tracked keypoints are described on the raw image, new ones
    are detected in the cells the tracks left empty (roi = the calibration's 5 px border), described and added with new map-point ids.
    Keypoints, ids, descriptors and the adapted detector state equal the oracle's composition of its numpy restatements."""
    from oracle import image_ref as R
    im = synth.make_pair(100 + detector, w, h)[0]
    rng = np.random.default_rng(4)
    first = R.detect_grid_fast_nosubpix(im, cs, np.zeros((0, 2)), 10, use_cv2=False)[0].astype(np.float32)
    tracked = np.ascontiguousarray(first[::4] + rng.uniform(-0.4, 0.4, first[::4].shape).astype(np.float32))
    cap = 4096
    lmid, px, desc, has = np.zeros(cap, np.int32), np.zeros((cap, 2), np.float32), np.zeros((cap, 32), np.uint8), np.zeros(cap, np.uint8)
    th, q = C.c_int(), C.c_double()
    K = np.array([458.654, 457.296, 367.215, 248.375])
    lib.ov2ref_extract_keypoints.restype = C.c_int
    n = lib.ov2ref_extract_keypoints(im.ctypes.data_as(U), im.ctypes.data_as(U), h, w, K.ctypes.data_as(D), cs, detector, 10, C.c_double(0.001),
                                     tracked.ctypes.data_as(C.POINTER(C.c_float)), len(tracked), cap, lmid.ctypes.data_as(I), px.ctypes.data_as(C.POINTER(C.c_float)),
                                     desc.ctypes.data_as(U), has.ctypes.data_as(U), C.byref(th), C.byref(q))
    assert len(tracked) < n <= cap
    roi = (5, 5, w - 10, h - 10)                                  # CameraCalibration's roi_rect_ (camera_calibration.cpp:72-73)
    if detector == 0:
        ipts, want_th, _ = R.detect_grid_fast_nosubpix(im, cs, tracked, 10, use_cv2=False)
        assert th.value == want_th
    else:
        ipts, want_q, _ = R.detect_single_scale_nosubpix(im, cs, tracked, roi, 0.001, use_cv2=False)
        assert q.value == want_q
    new = R.corner_subpix_cv2(im, ipts.astype(np.float32)) if len(ipts) else np.zeros((0, 2), np.float32)
    want_px = np.concatenate([tracked, new])
    assert n == len(want_px) and np.array_equal(lmid[:n], np.arange(n))        # tracked keep ids 0 .., new keypoints get the next ids in order
    assert np.array_equal(px[:n], want_px)
    wd, wv = R.describe_ref(im, want_px)
    assert np.array_equal(has[:n], wv) and np.array_equal(desc[:n][wv > 0], wd[wv > 0])


def test_ceres_pnp_equals_the_reference_function(lib):
    """The REFERENCE'S OWN MultiViewGeometry::ceresPnP (src/multi_view_geometry.cpp:492-588) - the function the drop-in
    host/multi_view_geometry_pnp_gpu.cpp replaces - on small problems (its 5 ms wall-clock cap must not bind on this build): verdict,
    rejected blocks and pose of oracle/pnp_ref.py::ceres_pnp."""
    from oracle import pnp_ref as P
    K32 = np.array([458.654, 457.296, 367.215, 248.375], np.float32)
    K = K32.astype(np.float64)
    rng = np.random.default_rng(12)
    lib.ov2ref_real_ceres_pnp.restype = C.c_int
    for case in range(6):
        n = 40 + 10 * case
        q = B.quat_normalize(np.array([0.0, 0.0, 0.0, 1.0]) + rng.normal(0, 0.1, 4))
        Ttrue = np.concatenate([rng.normal(0, 0.5, 3), q])
        pc = np.stack([rng.uniform(-2, 2, n), rng.uniform(-1.5, 1.5, n), rng.uniform(2, 10, n)], 1)
        w = np.ascontiguousarray(pc @ B.quat_to_rot(q).T + Ttrue[:3])
        px = np.stack([K[0] * pc[:, 0] / pc[:, 2] + K[2], K[1] * pc[:, 1] / pc[:, 2] + K[3]], 1) + rng.normal(0, 0.5, (n, 2))
        nbad = n // 8 if case % 2 else 0
        px[:nbad] += rng.uniform(15, 50, (nbad, 2))
        px = np.ascontiguousarray(px)
        scales = rng.integers(0, 3, n).astype(np.int32)
        T0 = B.pose_plus(Ttrue, np.concatenate([rng.normal(0, 0.04, 3), rng.normal(0, 0.015, 3)]))
        ok, pose, outliers = P.ceres_pnp(px, w, T0.copy(), K, nmaxiter=5, chi2th=5.9915, use_robust=True, apply_l2_after_robust=True, scales=scales)
        for attempt in range(4):            # the reference's cap is on wall-clock time: a solve cut short on a busy machine is retried
            T = T0.copy()
            out, nout = np.zeros(n, np.int32), C.c_int()
            rc = lib.ov2ref_real_ceres_pnp(n, px.ctypes.data_as(D), w.ctypes.data_as(D), scales.ctypes.data_as(I), T.ctypes.data_as(D), 5, C.c_float(5.9915), 1, 1,
                                           K32.ctypes.data_as(C.POINTER(C.c_float)), out.ctypes.data_as(I), C.byref(nout))
            if bool(rc) == ok and np.array_equal(out[:nout.value], outliers) and np.abs(T - pose).max() <= 1e-9:
                break
        else:
            raise AssertionError((case, rc, ok, np.abs(T - pose).max()))
