"""The drop-in C++ classes (ov2slam_b200/host/) behave like the Python binding of the same C ABI:
CPU part = they compile and link; GPU part = same keypoints / descriptors / tracks."""
import os
import subprocess
from pathlib import Path

import numpy as np
import pytest

from ov2slam_b200 import api, build, synth
from oracle import image_ref as R_img

ROOT = Path(__file__).resolve().parents[1]


def test_host_shims_compile_and_link():
    exe = build.build_host_shims()
    assert exe.exists()


@pytest.mark.gpu
def test_host_shims_match_python_binding(ctx, tmp_path):
    exe = build.build_host_shims()
    w, h = 640, 480
    prev, cur, _ = synth.make_pair(77, w, h)
    (tmp_path / "p.raw").write_bytes(prev.tobytes())
    (tmp_path / "c.raw").write_bytes(cur.tobytes())
    out = subprocess.run([str(exe), str(tmp_path / "p.raw"), str(tmp_path / "c.raw"), str(w), str(h)],
                         capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stderr
    tok = out.stdout.split()
    got = dict(nkps=int(tok[1]), th=int(tok[3]), kx=float(tok[5]), ky=float(tok[6]), ndesc=int(tok[8]), dsum=int(tok[10]),
               ngood=int(tok[12]))
    pp = api.Pyramid(ctx, 1, w, h, 3)
    cp = api.Pyramid(ctx, 1, w, h, 3)
    pp.build(prev[None])
    cp.build(cur[None])
    fe = api.FeatureExtractor(ctx, nfast_th=10)
    pts, _ = fe.detect_grid_fast_frame(pp, 0, 50, np.zeros((0, 2), np.float32))
    d = np.zeros((len(pts), 32), np.uint8)
    v = np.zeros(len(pts), np.uint8)
    fe.describe_brief(pp, pts, d, v)
    pri = pts.copy()
    st = np.zeros(len(pts), np.uint8)
    api.FeatureTracker(ctx, 30, 0.01).fb_klt_tracking(pp, cp, 9, 3, 30.0, 0.5, pts, pri, st)
    assert got["nkps"] == len(pts) and got["th"] == fe.nfast_th_
    assert abs(got["kx"] - float(pts[:, 0].astype(np.float64).sum())) < 1e-2
    assert got["ndesc"] == int(v.sum())
    assert got["dsum"] == int((d[v.astype(bool)].astype(np.int64) * np.arange(1, 33)).sum())
    assert got["ngood"] == int(st.sum())


_rect_subpix_template = R_img.get_rect_subpix_u8_ref
_line_min_sad_ref = R_img.line_min_sad_ref


def test_get_line_min_sad_matches_the_reference_function():
    """The drop-in FeatureTracker::getLineMinSAD (host C++) against a restatement of the reference's function with
    OpenCV's 8-bit getRectSubPix template: identical priors and errors - sub-pixel points, border window shrink, both
    scan directions (round 1 rounded the point, scanned the other way and dropped the shrink rule: ADVICE r1).  With
    cv2's own getRectSubPix (an IPP build: +-1 grey level on ~0.7 % of the pixels) the errors agree to 0.05 and the
    priors almost always."""
    exe = build.build_host_shims()
    w, h = 320, 240
    left = synth.make_frame(5, w, h, nrect=60)
    right = np.ascontiguousarray(np.roll(left, -7, axis=1))
    rng = np.random.default_rng(3)
    pts = [(rng.uniform(0, w - 1), rng.uniform(0, h - 1), 7, int(rng.integers(0, 2))) for _ in range(40)]
    pts += [(2.3, 100.7, 7, 1), (w - 2.2, 50.1, 7, 0), (150.5, 1.4, 7, 1), (150.5, h - 1.6, 7, 0), (60.0, 60.0, 8, 1), (0.4, 0.3, 7, 1)]
    import tempfile
    with tempfile.TemporaryDirectory() as d:
        (open(f"{d}/l.raw", "wb")).write(left.tobytes())
        (open(f"{d}/r.raw", "wb")).write(right.tobytes())
        args = [str(exe), "--sad", f"{d}/l.raw", f"{d}/r.raw", str(w), str(h), str(len(pts))]
        for x, y, ws, gl in pts:
            args += [repr(float(np.float32(x))), repr(float(np.float32(y))), str(ws), str(gl)]
        out = subprocess.run(args, capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stderr
    got = [tuple(float(v) for v in line.split()) for line in out.stdout.strip().splitlines()]
    assert len(got) == len(pts)
    try:
        import cv2
        cv_sub = lambda im, ws, cx, cy: cv2.getRectSubPix(im, (ws, ws), (float(cx), float(cy)))
    except Exception:
        cv_sub = None
    agree = 0
    for (x, y, ws, gl), (gx, ge) in zip(pts, got):
        rx, re = _line_min_sad_ref(left, right, (x, y), ws, bool(gl), _rect_subpix_template)
        if re is None:
            assert gx == -1.0
            continue
        assert np.float32(gx) == np.float32(rx) and np.float32(ge) == np.float32(re), ((x, y, ws, gl), (gx, ge), (rx, re))
        if cv_sub is not None:
            cx, ce = _line_min_sad_ref(left, right, (x, y), ws, bool(gl), cv_sub)
            assert abs(ge - ce) <= 0.05
            agree += np.float32(gx) == np.float32(cx)
    if cv_sub is not None:
        assert agree >= 0.8 * len(pts)


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


def _drop_landmarks_seen_only_by_constant_keyframes(pb):
    """Optimizer::localBA collects its landmarks from the 3D keypoints of the OPTIMISED keyframes (optimizer.cpp:178-180): a
    landmark whose anchor and observers are all constant keyframes is not part of the reference's window."""
    const = pb["pose_const"].astype(bool)
    npts = len(pb["lm_invdepth"])
    seen = ~const[pb["lm_anchor_cam"]]
    np.logical_or.at(seen, pb["obs_lm"], ~const[pb["obs_cam"]])
    keep_l = np.nonzero(seen)[0]
    remap = -np.ones(npts, np.int64)
    remap[keep_l] = np.arange(len(keep_l))
    keep_o = np.nonzero(seen[pb["obs_lm"]])[0]
    out = dict(pb)
    for k in ("lm_anchor_cam", "lm_anchor_px", "lm_invdepth"):
        out[k] = np.ascontiguousarray(pb[k][keep_l])
    for k in ("obs_cam", "obs_px") + (("obs_type",) if pb.get("obs_type") is not None else ()):
        out[k] = np.ascontiguousarray(pb[k][keep_o])
    out["obs_lm"] = np.ascontiguousarray(remap[pb["obs_lm"][keep_o]].astype(np.int32))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("stereo,stop", [(False, False), (True, False), (False, True)])
def test_optimizer_localba_shim_updates_the_map_like_the_flat_solve(ctx, tmp_path, stereo, stop):
    """The drop-in Optimizer::localBA (host/optimizer_localba_gpu.cpp, compiled against the stand-in map classes) on a
    synthetic map: window selection over the covisibility map, anchored inverse-depth flattening (mono / stereo), GPU solve,
    write-back - the keyframe poses and landmark inverse depths left in the map equal ov2_localba_solve on the flat window;
    a stop request raised before the call skips the refinement and is consumed (ADVICE r1: bstop_localba_ was never cleared)."""
    exe = build.build_optimizer_shim()
    pb = _drop_landmarks_seen_only_by_constant_keyframes(synth.make_ba_problem(61 + stereo, 9, 600, 2400, stereo=stereo))
    _write_window(tmp_path / "w.bin", pb)
    out = subprocess.run([str(exe), str(tmp_path / "w.bin"), str(tmp_path / "r.bin")] + (["stop"] if stop else []),
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stdout + out.stderr
    ncam, npts = len(pb["pose"]), len(pb["lm_invdepth"])
    raw = np.fromfile(tmp_path / "r.bin", np.uint8)
    pose = raw[:ncam * 56].view(np.float64).reshape(ncam, 7)
    invd = raw[ncam * 56:ncam * 56 + npts * 8].view(np.float64)
    ref = {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in pb.items()}
    if stop:
        api.request_stop_local_ba(ctx, True)
    res, flags = api.Optimizer(ctx).local_ba(ref)
    api.request_stop_local_ba(ctx, False)
    if stop:
        assert res["iters_refine"] == 0
    # the shim stores unit quaternions through Sophus (sign / normalisation): compare rotations up to sign
    for c in range(ncam):
        assert np.abs(pose[c, :3] - ref["pose"][c, :3]).max() <= 1e-7
        q, r = pose[c, 3:], ref["pose"][c, 3:] / np.linalg.norm(ref["pose"][c, 3:])
        assert min(np.abs(q - r).max(), np.abs(q + r).max()) <= 1e-7
    alive = invd >= 0
    assert alive.mean() > 0.9
    assert np.abs(invd[alive] - ref["lm_invdepth"][alive]).max() <= 1e-7


@pytest.mark.gpu
@pytest.mark.parametrize("mode,stereo", [("loose", False), ("loose", True), ("full", False), ("full", True)])
def test_optimizer_loose_and_full_ba_shims(ctx, tmp_path, mode, stereo):
    """8f-4: the drop-in Optimizer::looseBA / fullBA (optimizer.cpp:900-1671 / 1674-2331; same residual blocks as localBA over a
    keyframe RANGE: the first two (mono) / one (stereo) keyframes constant, all others optimised, one 5-iteration solve with
    function_tolerance 1e-4 for looseBA, up to 100 + 100 iterations at Ceres' default 1e-6 for fullBA) on a synthetic map:
    the map they leave behind equals ov2_localba_solve on the flat window with those options; looseBA also moves the current
    frame rigidly with the loop keyframe (checked inside the self-test)."""
    exe = build.build_optimizer_shim()
    pb = synth.make_ba_problem(71 + stereo, 9, 600, 2400, stereo=stereo)
    pb["pose_const"] = np.zeros_like(pb["pose_const"])
    pb["pose_const"][:1 if stereo else 2] = 1
    pb = _drop_landmarks_seen_only_by_constant_keyframes(pb)
    _write_window(tmp_path / "w.bin", pb)
    out = subprocess.run([str(exe), str(tmp_path / "w.bin"), str(tmp_path / "r.bin"), mode], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stdout + out.stderr
    ncam, npts = len(pb["pose"]), len(pb["lm_invdepth"])
    raw = np.fromfile(tmp_path / "r.bin", np.uint8)
    pose = raw[:ncam * 56].view(np.float64).reshape(ncam, 7)
    invd = raw[ncam * 56:ncam * 56 + npts * 8].view(np.float64)
    ref = {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in pb.items()}
    if mode == "loose":
        res, flags = api.Optimizer(ctx).local_ba(ref, max_iters_robust=5, max_iters_refine=0, function_tolerance=1e-4, apply_l2_after_robust=0)
        assert res["iters_refine"] == 0
    else:
        res, flags = api.Optimizer(ctx).local_ba(ref, max_iters_robust=100, max_iters_refine=100, function_tolerance=1e-6)
    assert res["final_cost"] < res["initial_cost"]
    for c in range(ncam):
        assert np.abs(pose[c, :3] - ref["pose"][c, :3]).max() <= 1e-7
        q, r = pose[c, 3:], ref["pose"][c, 3:] / np.linalg.norm(ref["pose"][c, 3:])
        assert min(np.abs(q - r).max(), np.abs(q + r).max()) <= 1e-7
    alive = invd >= 0
    assert alive.mean() > 0.9
    assert np.abs(invd[alive] - ref["lm_invdepth"][alive]).max() <= 1e-6 * np.abs(ref["lm_invdepth"][alive]).max() + 1e-7


# ---------------------------------------------------------------------------------------------- Mapper::matchToMap drop-in
def _write_match_scene(path, sc):
    hd = np.array([len(sc["kp_px"]), len(sc["mp_xyz"]), len(sc["desc"]), len(sc["obs_kf"]), len(sc["kf_Tcw"]), len(sc["cand_mp"]),
                   len(sc["cell_ptr"]) - 1, sc["nbwcells"], sc["ncellsize"], sc["img_w"], sc["img_h"], sc["dist"] is not None], np.int32)
    dist = np.zeros(5) if sc["dist"] is None else np.asarray(sc["dist"], np.float64)
    with open(path, "wb") as f:
        f.write(hd.tobytes())
        for a, t in ((sc["K"], np.float64), (dist, np.float64), (sc["Tcw"], np.float64), (sc["kf_Tcw"], np.float64), (sc["mp_xyz"], np.float64),
                     (sc["kp_px"], np.float32), (sc["obs_px"], np.float32), (sc["cell_ptr"], np.int32), (sc["cell_kp"], np.int32),
                     (sc["kp_lm"], np.int32), (sc["mp_desc_ptr"], np.int32), (sc["mp_obs_ptr"], np.int32), (sc["obs_kf"], np.int32),
                     (sc["cand_mp"], np.int32), (sc["desc"], np.uint8)):
            f.write(np.ascontiguousarray(a, t).tobytes())


def _read_match_result(path):
    raw = np.fromfile(path, np.int32)
    n = int(raw[0])
    order = raw[1:1 + n]
    m = int(raw[1 + n])
    pairs = raw[2 + n:2 + n + 2 * m].reshape(m, 2)
    return order, {(int(a), int(b)) for a, b in pairs}, int(raw[2 + n + 2 * m])


def _read_match_dump(path):
    raw = np.fromfile(path, np.uint8)
    hd = raw[:48].view(np.int32)
    nkps, nmps, ndesc, nobs, nkfs, ncand, ncells, nbw, cs, w, h, has_dist = (int(v) for v in hd)
    fl = raw[48:60].view(np.float32)
    off = [60]

    def take(n, t):
        b = n * np.dtype(t).itemsize
        a = raw[off[0]:off[0] + b].view(t).copy()
        off[0] += b
        return a
    sc = dict(img_w=w, img_h=h, ncellsize=cs, nbwcells=nbw, dmaxpxdist=fl[0], fdistratio=fl[1], view_th=fl[2])
    sc["K"] = take(4, np.float64)
    d = take(5, np.float64)
    sc["dist"] = d if has_dist else None
    sc["Tcw"] = take(12, np.float64)
    sc["kf_Tcw"] = take(12 * nkfs, np.float64).reshape(nkfs, 12)
    sc["mp_xyz"] = take(3 * nmps, np.float64).reshape(nmps, 3)
    sc["kp_px"] = take(2 * nkps, np.float32).reshape(nkps, 2)
    sc["obs_px"] = take(2 * nobs, np.float32).reshape(nobs, 2)
    sc["cell_ptr"] = take(ncells + 1, np.int32)
    sc["cell_kp"] = take(int(sc["cell_ptr"][-1]), np.int32)
    sc["kp_lm"] = take(nkps, np.int32)
    sc["mp_desc_ptr"] = take(nmps + 1, np.int32)
    sc["mp_obs_ptr"] = take(nmps + 1, np.int32)
    sc["obs_kf"] = take(nobs, np.int32)
    sc["cand_mp"] = take(ncand, np.int32)
    sc["mp_kfmask"] = take(4 * nmps, np.uint64).reshape(nmps, 4)
    sc["desc"] = take(32 * ndesc, np.uint8).reshape(ndesc, 32)
    assert off[0] == len(raw)
    return sc


def _match_pairs_by_identity(sc, kp_match):
    """(keypoint, map point) pairs named by what they ARE (pixel + own map point's position; candidate's position), so that two
    flattenings of the same map with different index orders can be compared."""
    out = set()
    for j, c in enumerate(kp_match):
        if c >= 0:
            out.add((tuple(sc["kp_px"][j]), tuple(sc["mp_xyz"][sc["kp_lm"][j]]), tuple(sc["mp_xyz"][sc["cand_mp"][c]])))
    return out


@pytest.mark.parametrize("distorted", [True, False])
def test_mapper_match_shim_flattens_the_map_like_the_scene(tmp_path, distorted):
    """The drop-in Mapper::matchToMap (host/mapper_match_gpu.cpp, against the stand-in map classes) on a synthetic map, with the
    GPU call replaced by a recorder (tests/helpers/match_dump.c, LD_PRELOAD): the flat problem it builds from the frame grid, the
    keyframes and the map points gives, through the oracle, the matches of the scene the map was built from (candidates in the
    order the shim walked the id set); map points without descriptor are filtered, keypoints whose map point is gone are dropped
    from the map (mapper.cpp:667-672), the search radius doubles for a frame with fewer than 30 3-D keypoints."""
    from oracle import match_ref as M
    exe = build.build_mapper_shim()
    rec = tmp_path / "librec.so"
    subprocess.check_call(["gcc", "-shared", "-fPIC", "-O1", "-o", str(rec), str(ROOT / "tests" / "helpers" / "match_dump.c")])
    sc = synth.make_match_scene(5 + distorted, nkps=500, ncand=260, nkfs=9, distorted=distorted)
    _write_match_scene(tmp_path / "s.bin", sc)
    env = dict(os.environ, LD_PRELOAD=str(rec), OV2_MATCH_DUMP=str(tmp_path / "d.bin"))
    out = subprocess.run([str(exe), str(tmp_path / "s.bin"), str(tmp_path / "r.bin")], capture_output=True, text=True, timeout=120, env=env)
    assert out.returncode == 0, out.stdout + out.stderr
    order, pairs, ndropped = _read_match_result(tmp_path / "r.bin")
    assert not pairs and ndropped == int((sc["kp_lm"] < 0).sum())
    dump = _read_match_dump(tmp_path / "d.bin")
    assert dump["dmaxpxdist"] == sc["dmaxpxdist"] and dump["fdistratio"] == sc["fdistratio"]
    assert abs(float(dump["view_th"]) - float(sc["view_th"])) <= 1e-6
    ndesc_of = np.diff(sc["mp_desc_ptr"])
    assert len(dump["cand_mp"]) == int((ndesc_of[sc["cand_mp"]] > 0).sum())
    ref = dict(sc, cand_mp=np.asarray(order, np.int32))
    want = _match_pairs_by_identity(ref, M.match_to_map(ref)[2])
    got = _match_pairs_by_identity(dump, M.match_to_map(dump)[2])
    assert len(want) > 40
    # poses travel through unit quaternions (as in the reference's map): last-bit differences in the projections
    assert len(want ^ got) <= max(1, len(want) // 100)


@pytest.mark.gpu
def test_mapper_match_shim_matches_python_binding(ctx, tmp_path):
    """The same drop-in end to end on the GPU: the (keypoint id -> map-point id) map it returns equals ov2_match_to_map on the scene
    the map was built from, candidates in the order the shim walked the id set."""
    exe = build.build_mapper_shim()
    sc = synth.make_match_scene(9, nkps=1200, ncand=700, nkfs=12, distorted=True)
    _write_match_scene(tmp_path / "s.bin", sc)
    out = subprocess.run([str(exe), str(tmp_path / "s.bin"), str(tmp_path / "r.bin")], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stdout + out.stderr
    order, pairs, _ = _read_match_result(tmp_path / "r.bin")
    ref = dict(sc, cand_mp=np.asarray(order, np.int32))
    _, _, kp_match, _ = api.match_to_map(ctx, ref)
    want = {(int(sc["kp_lm"][j]), int(order[c])) for j, c in enumerate(kp_match) if c >= 0}
    assert len(want) > 100
    assert len(want ^ pairs) <= max(1, len(want) // 100)


# ---------------------------------------------------------------------------------------------- MapManager::stereoMatching drop-in
def _quat_of(R):
    """Unit quaternion (x, y, z, w) of a rotation matrix with positive trace (small rotations only)."""
    w = 0.5 * np.sqrt(1.0 + np.trace(R))
    return np.array([(R[2, 1] - R[1, 2]) / (4 * w), (R[0, 2] - R[2, 0]) / (4 * w), (R[1, 0] - R[0, 1]) / (4 * w), w])


def _stereo_scene(seed, rect, nkps=320, w=752, h=480, cs=35, depth=None):
    rng = np.random.default_rng(seed)
    K = np.array([458.654, 457.296, 367.215, 248.375])
    Rrig = np.eye(3) if rect else synth._so3_exp(np.array([0.004, -0.006, 0.003]))
    trig = np.array([0.11, 0.0, 0.0]) if rect else np.array([0.11, 0.002, -0.001])        # right camera in the left camera's frame
    Rwc, twc = synth._so3_exp(rng.normal(0, 0.2, 3)), rng.normal(0, 1.0, 3)
    px = np.stack([rng.uniform(4, w - 4, nkps), rng.uniform(4, h - 4, nkps)], 1).astype(np.float32)
    bv = np.stack([(px[:, 0].astype(np.float64) - K[2]) / K[0], (px[:, 1].astype(np.float64) - K[3]) / K[1], np.ones(nkps)], 1)
    bv /= np.linalg.norm(bv, axis=1, keepdims=True)
    is3d = rng.random(nkps) < 0.6
    has_mp = is3d & (rng.random(nkps) > 0.08)
    z = rng.uniform(0.8, 8.0, nkps)
    cam = bv / bv[:, 2:3] * z[:, None] + rng.normal(0, 0.002, (nkps, 3))
    if depth is not None:
        cam = bv / bv[:, 2:3] * depth
    wpt = cam @ Rwc.T + twc
    # p_right = R_rl p_left + t_rl ;  F with  r^T F l = 0
    Rrl, trl = Rrig.T, -Rrig.T @ trig
    tx = np.array([[0, -trl[2], trl[1]], [trl[2], 0, -trl[0]], [-trl[1], trl[0], 0]])
    Kmat = np.array([[K[0], 0, K[2]], [0, K[1], K[3]], [0, 0, 1]])
    Frl = np.linalg.inv(Kmat).T @ tx @ Rrl @ np.linalg.inv(Kmat)
    return dict(rect=rect, w=w, h=h, cs=cs, nbw=int(np.ceil(w / cs)), nbh=int(np.ceil(h / cs)), K=K, Rrig=Rrig, trig=trig, Rwc=Rwc, twc=twc,
                Frl=Frl, lmid=(100 + np.arange(nkps)).astype(np.int32), is3d=is3d, has_mp=has_mp, px=px, unpx=px.copy(), bv=bv, wpt=wpt)


def _write_stereo_scene(path, sc):
    n = len(sc["lmid"])
    with open(path, "wb") as f:
        f.write(np.array([n, sc["rect"], sc["w"], sc["h"], sc["cs"], sc["nbw"], sc["nbw"] * sc["nbh"]], np.int32).tobytes())
        for a in (sc["K"], sc["K"], np.concatenate([sc["trig"], _quat_of(sc["Rrig"])]), np.concatenate([sc["twc"], _quat_of(sc["Rwc"])]), sc["Frl"]):
            f.write(np.ascontiguousarray(a, np.float64).tobytes())
        for i in range(n):
            f.write(np.array([sc["lmid"][i], sc["is3d"][i], sc["has_mp"][i]], np.int32).tobytes())
            f.write(np.concatenate([sc["px"][i], sc["unpx"][i]]).astype(np.float32).tobytes())
            f.write(np.concatenate([sc["bv"][i], sc["wpt"][i]]).astype(np.float64).tobytes())


def _read_mock_log(path):
    raw = np.fromfile(path, np.uint8)
    off, calls = 0, []
    while off < len(raw):
        tag = int(raw[off:off + 4].view(np.int32)[0])
        if tag == 3:
            calls.append(("build",))
            off += 4
        elif tag == 1:
            _, level, n, win, goleft = (int(v) for v in raw[off:off + 20].view(np.int32))
            pts = raw[off + 20:off + 20 + 8 * n].view(np.float32).reshape(n, 2).copy()
            calls.append(("sad", level, win, goleft, pts))
            off += 20 + 8 * n
        else:
            assert tag == 2
            _, n, nlv, win = (int(v) for v in raw[off:off + 16].view(np.int32))
            pts = raw[off + 16:off + 16 + 8 * n].view(np.float32).reshape(n, 2).copy()
            pri = raw[off + 16 + 8 * n:off + 16 + 16 * n].view(np.float32).reshape(n, 2).copy()
            calls.append(("klt", nlv, win, pts, pri))
            off += 16 + 16 * n
    return calls


def _mock_klt(pts, pri, nlv):
    """The canned tracker of tests/helpers/frontend_mock.c."""
    f32 = np.float32
    out = pri.copy()
    out[:, 0] += f32(-0.5)
    out[:, 1] += np.where(np.floor(pts[:, 0]).astype(int) % 7 == 0, f32(4.0), f32(0.25)).astype(np.float32)
    if nlv == 1:
        st = np.floor(f32(3.0) * pts[:, 0] + pts[:, 1]).astype(int) % 4 != 0
    else:
        st = np.floor(pts[:, 0] + f32(2.0) * pts[:, 1]).astype(int) % 6 != 0
    return out, st


def _mock_sad(sp):
    """The canned row search of tests/helpers/frontend_mock.c (coarsest-level pixels in, best column out)."""
    fx, fy = np.floor(sp[:, 0]).astype(int), np.floor(sp[:, 1]).astype(int)
    return np.where((fx >= 3) & (fy % 4 != 0), (fx - 2).astype(np.float32), np.float32(-1))


def _stereo_flow(sc, order, klt=None, sad=None):
    """MapManager::stereoMatching (map_manager.cpp:367-611) restated over the scene: the expected tracker / row-search calls and the
    expected stereo keypoints.  klt(pts, priors, nlevels) -> (moved priors, status) and sad(coarsest-level pts) -> columns default to the
    mock's rules; tests/test_oracle_vs_reference_map.py passes the real library's functions to compare with the reference's own code."""
    klt = klt or _mock_klt
    sad = sad or _mock_sad
    f32 = np.float32
    K, idx = sc["K"], {int(l): i for i, l in enumerate(sc["lmid"])}
    Rcw, Rrl = sc["Rwc"].T, sc["Rrig"].T

    def right_px(cam):
        p = Rrl @ (cam - sc["trig"])
        return np.array([f32(K[0] * p[0] / p[2] + K[2]), f32(K[1] * p[1] / p[2] + K[3])], np.float32)

    def in_right(p):
        return p[0] >= 0 and p[1] >= 0 and p[0] < sc["w"] and p[1] < sc["h"]
    cell = {}
    for i in range(len(sc["lmid"])):
        cell.setdefault((int(np.floor(sc["px"][i, 1] / f32(sc["cs"]))), int(np.floor(sc["px"][i, 0] / f32(sc["cs"])))), []).append(i)
    v3 = dict(ids=[], pts=[], pri=[])
    v2 = dict(ids=[], pts=[], pri=[])
    sad_pts, sad_slot, removed = [], [], 0
    for lm in order:
        i = idx[int(lm)]
        px = sc["px"][i]
        if sc["is3d"][i]:
            if sc["has_mp"][i]:
                proj = right_px(Rcw @ (sc["wpt"][i] - sc["twc"]))
                if in_right(proj):
                    v3["ids"].append(int(lm)); v3["pts"].append(px); v3["pri"].append(proj)
                    continue
            else:
                removed += 1
                continue
        if sc["rect"]:
            sad_pts.append(px * f32(0.125))
            sad_slot.append(len(v2["ids"]))
        else:
            r0, c0 = int(np.floor(px[1] / f32(sc["cs"]))), int(np.floor(px[0] / f32(sc["cs"])))
            nb, mean_z, wsum = 0, 0.0, 0.0
            for r in (r0 - 1, r0):
                for c in (c0 - 1, c0):
                    if r < 0 or c < 0 or r * sc["nbw"] + c >= sc["nbw"] * sc["nbh"]:
                        continue
                    for j in cell.get((r, c), []):
                        if j == i or not sc["is3d"][j] or not sc["has_mp"][j]:
                            continue
                        d = sc["unpx"][j] - sc["unpx"][i]
                        coef = 1.0 / np.sqrt(float(d[0]) ** 2 + float(d[1]) ** 2)
                        nb += 1
                        wsum += coef
                        mean_z += coef * (Rcw @ (sc["wpt"][j] - sc["twc"]))[2]
            if nb >= 1:
                proj = right_px(mean_z / wsum * (sc["bv"][i] / sc["bv"][i][2]))
                if in_right(proj):
                    v3["ids"].append(int(lm)); v3["pts"].append(px); v3["pri"].append(proj)
                    continue
        v2["ids"].append(int(lm)); v2["pts"].append(px); v2["pri"].append(px.copy())
    calls = []
    if sad_pts:
        sp = np.asarray(sad_pts, np.float32)
        calls.append(("sad", 3, 7, 1, sp))
        xpr = np.asarray(sad(sp), np.float32) * f32(8.0)
        for k, slot in enumerate(sad_slot):
            if xpr[k] >= 0 and xpr[k] <= v2["pts"][slot][0]:
                v2["pri"][slot][0] = xpr[k]
    good = []
    if v3["ids"]:
        pts, pri = np.asarray(v3["pts"], np.float32), np.asarray(v3["pri"], np.float32)
        calls.append(("klt", 1, 9, pts, pri))
        out, st = klt(pts, pri, 1)
        for k, lm in enumerate(v3["ids"]):
            if st[k]:
                good.append((lm, out[k]))
            else:
                v2["ids"].append(lm); v2["pts"].append(pts[k]); v2["pri"].append(out[k])
    if v2["ids"]:
        pts, pri = np.asarray(v2["pts"], np.float32), np.asarray(v2["pri"], np.float32)
        calls.append(("klt", 3, 9, pts, pri))
        out, st = klt(pts, pri, 3)
        good += [(lm, out[k]) for k, lm in enumerate(v2["ids"]) if st[k]]
    stereo = {}
    for lm, rp in good:
        lun = sc["unpx"][idx[lm]]
        rp = rp.copy()
        if sc["rect"]:
            err = abs(f32(lun[1] - rp[1]))
            rp[1] = lun[1]
        else:
            l, r = np.array([lun[0], lun[1], 1.0], np.float64), np.array([rp[0], rp[1], 1.0], np.float64)
            Fl, Ftr = sc["Frl"] @ l, sc["Frl"].T @ r
            err = np.sqrt(float(r @ Fl) ** 2 / (Ftr[0] ** 2 + Ftr[1] ** 2 + Fl[0] ** 2 + Fl[1] ** 2))
        if err <= 2.0:
            stereo[lm] = rp
    return calls, stereo, removed


@pytest.mark.parametrize("rect", [1, 0])
def test_stereo_matching_shim_flow(tmp_path, rect):
    """The drop-in MapManager::stereoMatching (host/map_manager_stereo_gpu.cpp + the drop-in FeatureTracker, against the stand-in map
    classes) on a synthetic stereo keyframe, with the device calls replaced by a recorder with rule-based answers
    (tests/helpers/frontend_mock.c, LD_PRELOAD): each image is uploaded once; rectified rigs make ONE batched row search on the
    coarsest level for exactly the keypoints without a usable map-point prior; the 2-level tracker call gets the projected /
    neighbour-depth priors, the full-pyramid call the rest plus the failed ones with their moved priors, in the reference's order;
    the epipolar test (row difference / Sampson distance) and the row correction decide the stereo keypoints the frame ends up with;
    keypoints whose map point is gone are dropped from the map."""
    exe = build.build_stereo_shim()
    mock = tmp_path / "libmock.so"
    subprocess.check_call(["gcc", "-shared", "-fPIC", "-O1", "-o", str(mock), str(ROOT / "tests" / "helpers" / "frontend_mock.c"), "-lm"])
    sc = _stereo_scene(31 + rect, rect)
    _write_stereo_scene(tmp_path / "s.bin", sc)
    env = dict(os.environ, LD_PRELOAD=str(mock), OV2_MOCK_LOG=str(tmp_path / "log.bin"))
    out = subprocess.run([str(exe), str(tmp_path / "s.bin"), str(tmp_path / "r.bin")], capture_output=True, text=True, timeout=120, env=env)
    assert out.returncode == 0, out.stdout + out.stderr
    raw = np.fromfile(tmp_path / "r.bin", np.uint8)
    n = int(raw[:4].view(np.int32)[0])
    order = raw[4:4 + 4 * n].view(np.int32)
    rec = raw[4 + 4 * n:4 + 16 * n].reshape(n, 12)
    is_stereo = rec[:, :4].copy().view(np.int32).reshape(n) != 0
    rpx = rec[:, 4:].copy().view(np.float32).reshape(n, 2)
    removed = int(raw[4 + 16 * n:].view(np.int32)[0])
    calls = _read_mock_log(tmp_path / "log.bin")
    want_calls, want_stereo, want_removed = _stereo_flow(sc, order)
    assert sum(c[0] == "build" for c in calls) == 2                      # left and right image: one upload each
    calls = [c for c in calls if c[0] != "build"]
    assert [c[:3] if c[0] == "klt" else c[:4] for c in calls] == [c[:3] if c[0] == "klt" else c[:4] for c in want_calls]
    assert len(calls) == (3 if rect else 2)
    for got, want in zip(calls, want_calls):
        for a, b in zip(got[3:] if got[0] == "klt" else got[4:], want[3:] if want[0] == "klt" else want[4:]):
            assert a.shape == b.shape and np.abs(a - b).max() <= 1e-3
    assert removed == want_removed and removed > 5
    got_ids = {int(l) for l, s in zip(order, is_stereo) if s}
    assert got_ids == set(want_stereo) and 60 < len(got_ids) < n - 40
    for l, p in zip(order, rpx):
        if int(l) in want_stereo:
            assert np.abs(p - want_stereo[int(l)]).max() <= 1e-3


@pytest.mark.gpu
def test_stereo_matching_shim_on_the_device(tmp_path):
    """The same drop-in end to end on the GPU, on a synthetic rectified pair (a smooth texture and its copy 16 px to the left = a
    fronto-parallel plane; map points on that plane): keypoints with a map point are tracked from their projected prior on two
    levels, the others from the batched row-search prior on the full pyramid; away from the left border nearly all become stereo
    keypoints 16 px to the left on the same row."""
    exe = build.build_stereo_shim()
    disp = 16.0
    K0, base = 458.654, 0.11
    sc = _stereo_scene(77, 1, depth=K0 * base / disp)
    _write_stereo_scene(tmp_path / "s.bin", sc)
    out = subprocess.run([str(exe), str(tmp_path / "s.bin"), str(tmp_path / "r.bin"), str(disp)], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stdout + out.stderr
    raw = np.fromfile(tmp_path / "r.bin", np.uint8)
    n = int(raw[:4].view(np.int32)[0])
    order = raw[4:4 + 4 * n].view(np.int32)
    rec = raw[4 + 4 * n:4 + 16 * n].reshape(n, 12)
    is_stereo = rec[:, :4].copy().view(np.int32).reshape(n) != 0
    rpx = rec[:, 4:].copy().view(np.float32).reshape(n, 2)
    idx = {int(l): i for i, l in enumerate(sc["lmid"])}
    px = np.stack([sc["px"][idx[int(l)]] for l in order])
    alive = np.array([not (sc["is3d"][idx[int(l)]] and not sc["has_mp"][idx[int(l)]]) for l in order])
    inner = alive & (px[:, 0] > 60) & (px[:, 0] < sc["w"] - 20) & (px[:, 1] > 20) & (px[:, 1] < sc["h"] - 20)
    assert inner.sum() > 150
    assert is_stereo[inner].mean() > 0.9, out.stdout + out.stderr
    err = np.abs(rpx[inner & is_stereo] - (px[inner & is_stereo] - np.array([disp, 0.0], np.float32)))
    assert np.median(err[:, 0]) < 0.05 and (err[:, 0] < 0.5).mean() > 0.97 and err[:, 1].max() == 0.0
    assert not is_stereo[~alive].any()


def test_clahe_adapter_routes_cv_clahe_calls_to_the_device_call(tmp_path):
    """The cv::CLAHE adapter (host/clahe_gpu.cpp; replaces the reference's one cv::createCLAHE call, ov2slam.cpp:87) with the device
    call mocked (dst = 255 - src): a ROI source (row step > width) into a fresh destination and an in-place call both reach
    ov2_clahe with the image size, ONE row stride valid for both buffers, clip limit 3 and the W/50 x H/50 tile grid; an empty
    image gives an empty result."""
    build.build_host_shims()
    exe = build.LIB / "clahe_selftest"
    mock = tmp_path / "libmock.so"
    subprocess.check_call(["gcc", "-shared", "-fPIC", "-O1", "-o", str(mock), str(ROOT / "tests" / "helpers" / "frontend_mock.c"), "-lm"])
    w, h = 173, 121
    env = dict(os.environ, LD_PRELOAD=str(mock), OV2_MOCK_LOG=str(tmp_path / "log.bin"))
    out = subprocess.run([str(exe), str(w), str(h), str(tmp_path / "o.bin")], capture_output=True, text=True, timeout=60, env=env)
    assert out.returncode == 0, out.stdout + out.stderr
    yy, xx = np.mgrid[0:h, 0:w]
    src = ((xx * 7 + yy * 13 + (xx * yy) % 5) & 255).astype(np.uint8)
    got = np.fromfile(tmp_path / "o.bin", np.uint8).reshape(2, h, w)
    assert np.array_equal(got[0], 255 - src) and np.array_equal(got[1], 255 - src)
    log = np.fromfile(tmp_path / "log.bin", np.int32).reshape(-1, 9)
    assert len(log) == 2 and (log[:, 0] == 4).all()
    for rec in log:
        assert tuple(rec[1:3]) == (w, h) and rec[3] == w and rec[4] == 1 and rec[5] == 3000 and tuple(rec[6:8]) == (w // 50, h // 50)
        assert rec[8] == 1          # both calls equalise in place in the destination's layout (the source was copied there first / is it)

