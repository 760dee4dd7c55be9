"""Seeded synthetic inputs for the two hot paths (SURVEY.md section 8d).

numpy only (no cv2) so the same bytes are produced here, on the GPU box, in the tests and in
bench.py.  Nothing in this file is on the product path; it only manufactures inputs.

  * make_frame / make_pair  - corner-rich 8-bit images and a (prev, cur) pair with known flow
  * make_ba_problem         - a synthetic local-BA window in the flat SoA layout the C ABI takes
                              (the flattening Optimizer::localBA's setup performs,
                              /root/reference/src/optimizer.cpp:43-430)
"""
from __future__ import annotations

import numpy as np


# ----------------------------------------------------------------------------- images
def _gauss_kernel(sigma: float) -> np.ndarray:
    r = int(np.ceil(3 * sigma))
    x = np.arange(-r, r + 1, dtype=np.float64)
    k = np.exp(-0.5 * (x / sigma) ** 2)
    return k / k.sum()


def _sep_blur(img: np.ndarray, sigma: float) -> np.ndarray:
    k = _gauss_kernel(sigma)
    r = len(k) // 2
    p = np.pad(img, ((r, r), (r, r)), mode="reflect")
    tmp = np.zeros((p.shape[0], img.shape[1]), np.float64)
    for i, kv in enumerate(k):
        tmp += kv * p[:, i:i + img.shape[1]]
    out = np.zeros(img.shape, np.float64)
    for i, kv in enumerate(k):
        out += kv * tmp[i:i + img.shape[0], :]
    return out


def make_frame(seed: int, w: int = 640, h: int = 480, nrect: int = 200) -> np.ndarray:
    """Blurred-noise texture (many FAST-10 corners per cell) + random grey rectangles
    (strong, response >= 20, corners).  Returns (h, w) uint8, C-contiguous."""
    rng = np.random.default_rng(seed)
    base = rng.integers(0, 256, size=(h, w)).astype(np.float64)
    base = _sep_blur(base, 2.0)
    base = (base - base.min()) / max(base.max() - base.min(), 1e-9) * 255.0
    for _ in range(nrect):
        rw = int(rng.integers(8, 64))
        rh = int(rng.integers(8, 64))
        x0 = int(rng.integers(-8, w - 8))
        y0 = int(rng.integers(-8, h - 8))
        g = float(rng.integers(0, 256))
        a = float(rng.uniform(0.55, 1.0))
        ys, ye = max(y0, 0), min(y0 + rh, h)
        xs, xe = max(x0, 0), min(x0 + rw, w)
        if ys < ye and xs < xe:
            base[ys:ye, xs:xe] = (1 - a) * base[ys:ye, xs:xe] + a * g
    base = _sep_blur(base, 0.7)
    return np.clip(np.rint(base), 0, 255).astype(np.uint8)


def shift_image(img: np.ndarray, dx: float, dy: float) -> np.ndarray:
    """cur(x, y) = img(x - dx, y - dy), bilinear, edge-replicated.  float64 result."""
    h, w = img.shape
    xs = np.arange(w, dtype=np.float64) - dx
    ys = np.arange(h, dtype=np.float64) - dy
    x0 = np.floor(xs).astype(np.int64)
    y0 = np.floor(ys).astype(np.int64)
    ax = (xs - x0)[None, :]
    ay = (ys - y0)[:, None]
    x0c = np.clip(x0, 0, w - 1)
    x1c = np.clip(x0 + 1, 0, w - 1)
    y0c = np.clip(y0, 0, h - 1)
    y1c = np.clip(y0 + 1, 0, h - 1)
    f = img.astype(np.float64)
    top = f[y0c][:, x0c] * (1 - ax) + f[y0c][:, x1c] * ax
    bot = f[y1c][:, x0c] * (1 - ax) + f[y1c][:, x1c] * ax
    return top * (1 - ay) + bot * ay


def make_pair(seed: int, w: int = 640, h: int = 480, max_shift: float = 8.0,
              noise_sigma: float = 2.0):
    """(prev, cur, flow): cur = prev translated by `flow` (px) + N(0, noise_sigma) noise."""
    prev = make_frame(seed, w, h)
    rng = np.random.default_rng(seed + 1_000_003)
    flow = rng.uniform(-max_shift, max_shift, size=2)
    cur = shift_image(prev, float(flow[0]), float(flow[1]))
    cur = cur + rng.normal(0.0, noise_sigma, size=cur.shape)
    cur = np.clip(np.rint(cur), 0, 255).astype(np.uint8)
    return prev, cur, flow.astype(np.float32)


def make_batch(first_seed: int, nframes: int, w: int = 640, h: int = 480):
    """Batch of independent (prev, cur) pairs: two (B, h, w) uint8 arrays + (B, 2) float32 flows."""
    prevs = np.empty((nframes, h, w), np.uint8)
    curs = np.empty((nframes, h, w), np.uint8)
    flows = np.empty((nframes, 2), np.float32)
    for i in range(nframes):
        prevs[i], curs[i], flows[i] = make_pair(first_seed + i, w, h)
    return prevs, curs, flows


def make_priors(seed: int, kps: np.ndarray, flow: np.ndarray, frac3d: float = 0.6):
    """Split keypoints the way VisualFrontEnd::kltTracking does
    (/root/reference/src/visual_front_end.cpp:156-251): a seeded `frac3d` subset gets a
    motion prior = true flow + N(0, 1) px and is tracked with nbpyrlvl = 1; the rest start from
    their previous position and use the full pyramid (nbpyrlvl = 3).
    Returns (is3d bool[N], priors float32[N, 2])."""
    rng = np.random.default_rng(seed + 7_000_003)
    n = len(kps)
    is3d = rng.random(n) < frac3d
    pri = kps.astype(np.float32).copy()
    jitter = rng.normal(0.0, 1.0, size=(n, 2)).astype(np.float32)
    pri[is3d] = (kps[is3d] + flow[None, :].astype(np.float32) + jitter[is3d]).astype(np.float32)
    return is3d, pri


# ----------------------------------------------------------------------------- local BA
def _so3_exp(w: np.ndarray) -> np.ndarray:
    th = np.linalg.norm(w)
    K = np.array([[0, -w[2], w[1]], [w[2], 0, -w[0]], [-w[1], w[0], 0]])
    if th < 1e-12:
        return np.eye(3) + K
    return np.eye(3) + np.sin(th) / th * K + (1 - np.cos(th)) / th ** 2 * (K @ K)


def _rot_to_quat_xyzw(R: np.ndarray) -> np.ndarray:
    t = np.trace(R)
    if t > 0:
        s = np.sqrt(t + 1.0) * 2
        q = np.array([(R[2, 1] - R[1, 2]) / s, (R[0, 2] - R[2, 0]) / s, (R[1, 0] - R[0, 1]) / s, 0.25 * s])
    else:
        i = int(np.argmax(np.diag(R)))
        j, k = (i + 1) % 3, (i + 2) % 3
        s = np.sqrt(1.0 + R[i, i] - R[j, j] - R[k, k]) * 2
        q = np.zeros(4)
        q[i] = 0.25 * s
        q[j] = (R[j, i] + R[i, j]) / s
        q[k] = (R[k, i] + R[i, k]) / s
        q[3] = (R[k, j] - R[j, k]) / s
    q = q / np.linalg.norm(q)
    if q[3] < 0:
        q = -q
    return q


def make_ba_problem(seed: int, ncam: int = 10, npts: int = 2000, nobs: int = 8000,
                    nconst: int = 2, outlier_frac: float = 0.05, px_noise: float = 0.5,
                    w: int = 752, h: int = 480, stereo: bool = False, baseline: float = 0.11):
    """Synthetic localBA window (SURVEY.md section 8d) as a dict of flat arrays:

      K[4]            fx, fy, cx, cy  (EuRoC, euroc_mono.yaml:21-24)
      pose[Nc, 7]     Twc as [tx, ty, tz, qx, qy, qz, qw]  (se3_param_block.hpp:39-46)
      pose_const[Nc]  1 = constant parameter block (gauge / non-optimised keyframe)
      lm_anchor_cam[Np], lm_anchor_px[Np, 2] (f64, values exactly representable in f32),
      lm_invdepth[Np]
      obs_cam[No], obs_lm[No], obs_px[No, 2]   non-anchor observations, sorted by landmark
      truth_pose / truth_invdepth             for convergence checks only

    Every landmark is anchored in its lowest-index observing camera; `nobs` counts the
    non-anchor observations (= residual blocks, the anchor observation itself carries no
    residual in the anchored inverse-depth parametrisation, optimizer.cpp:258-290).

    stereo=True adds, as the reference does for stereo keypoints (optimizer.cpp:270-330): one
    right-camera residual in the anchor frame (obs_type 2) and one right-camera residual next to
    every left-camera residual in the other frames (obs_type 1), a right calibration Kr and the
    constant extrinsic Trl (right-from-left; rectified rig, `baseline` metres along +x).  The
    residual-block count becomes npts + 2 * nobs.
    """
    rng = np.random.default_rng(seed)
    fx = fy = 458.654
    cx, cy = 367.215, 248.375
    K = np.array([fx, fy, cx, cy])
    # cameras on a smooth trajectory: 0.2 m steps along x, looking down +z, +-5 deg yaw jitter
    Rwc, twc = [], []
    for i in range(ncam):
        yaw = np.deg2rad(rng.uniform(-5, 5))
        Rwc.append(_so3_exp(np.array([0.0, yaw, 0.0])))
        twc.append(np.array([0.2 * i, rng.normal(0, 0.02), rng.normal(0, 0.02)]))
    Rwc = np.array(Rwc)
    twc = np.array(twc)

    def project(ci, pw):
        pc = Rwc[ci].T @ (pw - twc[ci])
        if pc[2] <= 0.5:
            return None
        u = fx * pc[0] / pc[2] + cx
        v = fy * pc[1] / pc[2] + cy
        if 5 <= u < w - 5 and 5 <= v < h - 5:
            return np.array([u, v]), pc[2]
        return None

    per_pt = nobs / npts  # mean number of non-anchor observations per landmark
    lm_anchor_cam = np.zeros(npts, np.int32)
    lm_anchor_px = np.zeros((npts, 2))
    lm_invdepth_true = np.zeros(npts)
    obs_cam, obs_lm, obs_px = [], [], []
    pi = 0
    target_counts = np.full(npts, int(np.floor(per_pt)), np.int64)
    extra = nobs - int(target_counts.sum())
    target_counts[rng.choice(npts, size=extra, replace=False)] += 1
    while pi < npts:
        # sample a point in front of a random camera
        c0 = int(rng.integers(0, ncam))
        z = rng.uniform(2.0, 15.0)
        u = rng.uniform(20, w - 20)
        v = rng.uniform(20, h - 20)
        pc = np.array([(u - cx) / fx * z, (v - cy) / fy * z, z])
        pw = Rwc[c0] @ pc + twc[c0]
        vis = [ci for ci in range(ncam) if project(ci, pw) is not None]
        need = int(target_counts[pi]) + 1
        if len(vis) < need:
            continue
        sel = np.sort(rng.choice(vis, size=need, replace=False))
        anch = int(sel[0])
        pa, za = project(anch, pw)
        # anchor pixel is stored as cv::Point2f in the reference: round to f32, and define the
        # true landmark as lying on that (rounded) bearing so the ground truth is consistent
        pa32 = pa.astype(np.float32).astype(np.float64)
        pc_a = np.array([(pa32[0] - cx) / fx * za, (pa32[1] - cy) / fy * za, za])
        pw = Rwc[anch] @ pc_a + twc[anch]
        lm_anchor_cam[pi] = anch
        lm_anchor_px[pi] = pa32
        lm_invdepth_true[pi] = 1.0 / za
        for ci in sel[1:]:
            pr = project(int(ci), pw)
            if pr is None:
                px = np.array([cx, cy])
            else:
                px = pr[0]
            px = px + rng.normal(0, px_noise, size=2)
            if rng.random() < outlier_frac:
                ang = rng.uniform(0, 2 * np.pi)
                px = px + rng.uniform(10, 50) * np.array([np.cos(ang), np.sin(ang)])
            obs_cam.append(int(ci))
            obs_lm.append(pi)
            obs_px.append(px.astype(np.float32).astype(np.float64))
        pi += 1

    truth_pose = np.zeros((ncam, 7))
    pose = np.zeros((ncam, 7))
    pose_const = np.zeros(ncam, np.uint8)
    pose_const[:nconst] = 1
    for i in range(ncam):
        truth_pose[i, :3] = twc[i]
        truth_pose[i, 3:] = _rot_to_quat_xyzw(Rwc[i])
        if pose_const[i]:
            pose[i] = truth_pose[i]
        else:
            dR = _so3_exp(rng.normal(0, np.deg2rad(0.5), size=3))
            pose[i, :3] = twc[i] + rng.normal(0, 0.01, size=3)
            pose[i, 3:] = _rot_to_quat_xyzw(dR @ Rwc[i])
    lm_invdepth = lm_invdepth_true * (1 + rng.normal(0, 0.05, size=npts))
    if stereo:
        Kr = K.copy()
        Trl = np.array([-baseline, 0.0, 0.0, 0.0, 0.0, 0.0, 1.0])
        o_cam, o_lm, o_px, o_typ = [], [], [], []
        mono_cam = np.array(obs_cam, np.int32)
        mono_lm = np.array(obs_lm, np.int32)
        mono_px = np.array(obs_px, np.float64).reshape(-1, 2)
        k = 0

        def right_px(pc):
            pr = pc + Trl[:3]
            uv = np.array([fx * pr[0] / pr[2] + cx, fy * pr[1] / pr[2] + cy]) + rng.normal(0, px_noise, size=2)
            if rng.random() < outlier_frac:
                ang = rng.uniform(0, 2 * np.pi)
                uv = uv + rng.uniform(10, 50) * np.array([np.cos(ang), np.sin(ang)])
            return uv.astype(np.float32).astype(np.float64)

        for l in range(npts):
            a = lm_anchor_cam[l]
            za = 1.0 / lm_invdepth_true[l]
            pc_a = np.array([(lm_anchor_px[l, 0] - cx) / fx * za, (lm_anchor_px[l, 1] - cy) / fy * za, za])
            pw = Rwc[a] @ pc_a + twc[a]
            o_cam.append(a); o_lm.append(l); o_px.append(right_px(pc_a)); o_typ.append(2)
            while k < len(mono_lm) and mono_lm[k] == l:
                c = int(mono_cam[k])
                o_cam.append(c); o_lm.append(l); o_px.append(mono_px[k]); o_typ.append(0)
                o_cam.append(c); o_lm.append(l); o_px.append(right_px(Rwc[c].T @ (pw - twc[c]))); o_typ.append(1)
                k += 1
        return dict(
            K=K, Kr=Kr, Trl=Trl, pose=pose, pose_const=pose_const,
            lm_anchor_cam=lm_anchor_cam, lm_anchor_px=lm_anchor_px, lm_invdepth=lm_invdepth,
            obs_cam=np.array(o_cam, np.int32), obs_lm=np.array(o_lm, np.int32),
            obs_px=np.array(o_px, np.float64).reshape(-1, 2), obs_type=np.array(o_typ, np.uint8),
            truth_pose=truth_pose, truth_invdepth=lm_invdepth_true,
        )
    return dict(
        K=K, pose=pose, pose_const=pose_const,
        lm_anchor_cam=lm_anchor_cam, lm_anchor_px=lm_anchor_px, lm_invdepth=lm_invdepth,
        obs_cam=np.array(obs_cam, np.int32), obs_lm=np.array(obs_lm, np.int32),
        obs_px=np.array(obs_px, np.float64).reshape(-1, 2),
        truth_pose=truth_pose, truth_invdepth=lm_invdepth_true,
    )


def make_loop_ba_problem(seed: int, nkf: int = 160, npts: int = 8000, obs_per_pt: int = 5, outlier_frac: float = 0.05,
                         px_noise: float = 0.5, w: int = 752, h: int = 480, stereo: bool = False, baseline: float = 0.11,
                         nconst_extra: int = 0, step: float = 0.2):
    """A long BA window over a CLOSED trajectory (loop-closure looseBA / fullBA sizes), vectorised, in the conventions of
    make_ba_problem: anchor = lowest-index observer, observations sorted by landmark (non-anchor views in ascending
    keyframe order), f32-representable pixels, truth_pose / truth_invdepth, the first 2 (mono) / 1 (stereo) keyframes
    constant, stereo residual types 2 / 0 / 1 as make_ba_problem lays them out.

    `nkf` keyframes sit on a circle (`step` metres apart) looking outwards; a landmark is seen by `obs_per_pt` + 1
    consecutive keyframes, so the reduced camera system is a band, and the landmarks around the start are seen by the last
    keyframes as well: the loop-closure blocks.  `nconst_extra` constant keyframes (a second pass half a step off the first)
    are appended after the `nkf`; each sees the landmarks in front of it once more (windows with more than 256 keyframes in
    total)."""
    rng = np.random.default_rng(seed)
    fx = fy = 458.654
    cx, cy = 367.215, 248.375
    K = np.array([fx, fy, cx, cy])
    R0 = nkf * step / (2 * np.pi)

    def rig(theta, y):
        c, s_ = np.cos(theta), np.sin(theta)
        Rwc = np.zeros((len(theta), 3, 3))
        Rwc[:, :, 0] = np.stack([s_, np.zeros_like(c), -c], 1)     # x: tangent
        Rwc[:, 1, 1] = 1.0                                            # y: world y
        Rwc[:, :, 2] = np.stack([c, np.zeros_like(c), s_], 1)      # z: outwards
        twc = np.stack([R0 * c, y, R0 * s_], 1)
        return Rwc, twc

    th = 2 * np.pi * np.arange(nkf) / nkf
    Rwc, twc = rig(th + np.deg2rad(rng.uniform(-2, 2, nkf)), rng.normal(0, 0.02, nkf))
    Rx, tx = rig(2 * np.pi * (np.arange(nconst_extra) + 0.5) / max(nconst_extra, 1), np.full(nconst_extra, 0.05))
    Rall, tall = np.concatenate([Rwc, Rx]), np.concatenate([twc, tx])
    ncam = nkf + nconst_extra

    def project(ci, pw):                      # ci [M, k], pw [M, 3] -> px [M, k, 2], z [M, k]
        pc = np.einsum("mkji,mkj->mki", Rall[ci], pw[:, None, :] - tall[ci])
        z = pc[..., 2]
        zs = np.where(np.abs(z) > 1e-9, z, 1e-9)
        return np.stack([fx * pc[..., 0] / zs + cx, fy * pc[..., 1] / zs + cy], -1), z

    def visible(px, z):
        return (z > 0.5) & (px[..., 0] >= 5) & (px[..., 0] < w - 5) & (px[..., 1] >= 5) & (px[..., 1] < h - 5)

    k = obs_per_pt + 1
    pws, cams = [], []
    have = 0
    while have < npts:
        m = 2 * (npts - have) + 64
        c0 = rng.integers(0, nkf, m)
        run = (c0[:, None] + np.arange(k)[None, :]) % nkf                       # consecutive keyframes (wrapping: loop)
        mid = run[:, k // 2]
        pc = np.stack([rng.uniform(-2.5, 2.5, m), rng.uniform(-1.5, 1.5, m), rng.uniform(4.0, 12.0, m)], 1)
        pw = np.einsum("mij,mj->mi", Rall[mid], pc) + tall[mid]
        ok = visible(*project(run, pw)).all(1)
        pws.append(pw[ok]); cams.append(np.sort(run[ok], 1))
        have += int(ok.sum())
    pw = np.concatenate(pws)[:npts]
    sel = np.concatenate(cams)[:npts]
    anch = sel[:, 0]
    # anchor pixel rounded to f32 and the landmark put on that bearing (make_ba_problem's convention)
    pa, za = project(anch[:, None], pw)
    pa32 = pa[:, 0].astype(np.float32).astype(np.float64)
    za = za[:, 0]
    pc_a = np.stack([(pa32[:, 0] - cx) / fx * za, (pa32[:, 1] - cy) / fy * za, za], 1)
    pw = np.einsum("mij,mj->mi", Rall[anch], pc_a) + tall[anch]
    obs = sel[:, 1:]
    if nconst_extra > 0:
        ang = np.arctan2(pw[:, 2], pw[:, 0]) % (2 * np.pi)
        ex = nkf + (np.floor(ang / (2 * np.pi) * nconst_extra).astype(np.int64) % nconst_extra)
        okx = visible(*project(ex[:, None], pw))[:, 0]
        obs = np.concatenate([obs, np.where(okx, ex, -1)[:, None]], 1)
    lm = np.repeat(np.arange(npts), obs.shape[1])
    oc = obs.reshape(-1)
    keep = oc >= 0
    lm, oc = lm[keep], oc[keep]
    px, _ = project(oc[:, None], pw[lm])
    px = px[:, 0] + rng.normal(0, px_noise, (len(oc), 2))

    def outliers(p):
        bad = rng.random(len(p)) < outlier_frac
        ang_ = rng.uniform(0, 2 * np.pi, len(p))
        r = rng.uniform(10, 50, len(p))
        return p + bad[:, None] * r[:, None] * np.stack([np.cos(ang_), np.sin(ang_)], 1)

    px = outliers(px).astype(np.float32).astype(np.float64)
    truth_pose = np.zeros((ncam, 7))
    truth_pose[:, :3] = tall
    truth_pose[:, 3:] = np.array([_rot_to_quat_xyzw(R) for R in Rall])
    pose_const = np.zeros(ncam, np.uint8)
    pose_const[:1 if stereo else 2] = 1
    pose_const[nkf:] = 1
    pose = truth_pose.copy()
    for i in np.nonzero(pose_const == 0)[0]:
        dR = _so3_exp(rng.normal(0, np.deg2rad(0.5), size=3))
        pose[i, :3] = tall[i] + rng.normal(0, 0.01, size=3)
        pose[i, 3:] = _rot_to_quat_xyzw(dR @ Rall[i])
    lm_invdepth_true = 1.0 / za
    lm_invdepth = lm_invdepth_true * (1 + rng.normal(0, 0.05, size=npts))
    out = dict(K=K, pose=pose, pose_const=pose_const, lm_anchor_cam=anch.astype(np.int32), lm_anchor_px=pa32,
               lm_invdepth=lm_invdepth, truth_pose=truth_pose, truth_invdepth=lm_invdepth_true)
    if not stereo:
        out.update(obs_cam=oc.astype(np.int32), obs_lm=lm.astype(np.int32), obs_px=px)
        return out
    # stereo: per landmark [anchor right view (2)], then (left (0), right (1)) for every other view
    Trl = np.array([-baseline, 0.0, 0.0, 0.0, 0.0, 0.0, 1.0])

    def right_px(pc):
        pr = pc + Trl[:3]
        uv = np.stack([fx * pr[:, 0] / pr[:, 2] + cx, fy * pr[:, 1] / pr[:, 2] + cy], 1) + rng.normal(0, px_noise, (len(pc), 2))
        return outliers(uv).astype(np.float32).astype(np.float64)

    pcam = np.einsum("mji,mj->mi", Rall[oc], pw[lm] - tall[oc])
    r_other = right_px(pcam)
    r_anch = right_px(pc_a)
    cnt = np.bincount(lm, minlength=npts)
    start = np.concatenate([[0], np.cumsum(1 + 2 * cnt)])[:-1]                  # first row of each landmark
    j = np.arange(len(lm)) - np.concatenate([[0], np.cumsum(cnt)])[:-1][lm]      # rank of the view within its landmark
    nob = int((1 + 2 * cnt).sum())
    o_cam = np.zeros(nob, np.int32); o_lm = np.zeros(nob, np.int32); o_px = np.zeros((nob, 2)); o_ty = np.zeros(nob, np.uint8)
    o_cam[start] = anch; o_lm[start] = np.arange(npts); o_px[start] = r_anch; o_ty[start] = 2
    rl = start[lm] + 1 + 2 * j
    o_cam[rl] = oc; o_lm[rl] = lm; o_px[rl] = px; o_ty[rl] = 0
    o_cam[rl + 1] = oc; o_lm[rl + 1] = lm; o_px[rl + 1] = r_other; o_ty[rl + 1] = 1
    out.update(Kr=K.copy(), Trl=Trl, obs_cam=o_cam, obs_lm=o_lm, obs_px=o_px, obs_type=o_ty)
    return out


# ----------------------------------------------------------------------------- local-map matching scene (Mapper::matchToMap)
def _proj_radtan(P, K, dist):
    x, y = P[:, 0] / P[:, 2], P[:, 1] / P[:, 2]
    if dist is not None:
        k1, k2, p1, p2, k3 = dist
        r2 = x * x + y * y
        cd = 1 + k1 * r2 + k2 * r2 * r2 + k3 * r2 ** 3
        x, y = x * cd + 2 * p1 * x * y + p2 * (r2 + 2 * x * x), y * cd + p1 * (r2 + 2 * y * y) + 2 * p2 * x * y
    return np.stack([K[0] * x + K[2], K[1] * y + K[3]], 1)


def make_match_scene(seed: int, nkps: int = 800, ncand: int = 400, nkfs: int = 12, distorted: bool = True,
                     w: int = 752, h: int = 480, ncellsize: int = 35) -> dict:
    """A flattened Mapper::matchToMap problem (the arrays ov2_match_to_map takes): a frame with `nkps` keypoints in its grid
    (85 % of them attached to a map point), `nkfs` keyframes around it, and `ncand` local map points the frame does not
    observe - half of them near-duplicates of observed map points (close in space, descriptors a few bits apart, mostly seen
    from other keyframes), the rest unrelated.  Map points carry 1-4 descriptors and 1-5 keyframe observations."""
    rng = np.random.default_rng(seed)
    K = np.array([458.654, 457.296, 367.215, 248.375])
    dist = np.array([-0.28340811, 0.07395907, 0.00019359, 1.76187114e-05, 0.0]) if distorted else None

    def pose(scale):
        R = _so3_exp(rng.normal(0, 0.05 * scale, 3))
        t = rng.normal(0, 0.3 * scale, 3)
        return np.concatenate([R.reshape(-1), t])       # Tcw: camera <- world

    Tcw = pose(0.2)
    kf_T = np.stack([pose(1.0) for _ in range(nkfs)])
    R, t = Tcw[:9].reshape(3, 3), Tcw[9:]
    # observed map points: sample pixels, back-project at random depths into the world
    nobs_mp = int(0.85 * nkps)
    pix = np.stack([rng.uniform(5, w - 5, nkps), rng.uniform(5, h - 5, nkps)], 1)
    z = rng.uniform(2.0, 10.0, nkps)
    cam = np.stack([(pix[:, 0] - K[2]) / K[0] * z, (pix[:, 1] - K[3]) / K[1] * z, z], 1)
    world = (cam - t) @ R                                  # R^T (cam - t)
    kp_px = _proj_radtan(world @ R.T + t, K, dist).astype(np.float32)
    inimg = (kp_px[:, 0] >= 0) & (kp_px[:, 1] >= 0) & (kp_px[:, 0] < w) & (kp_px[:, 1] < h)
    kp_px[~inimg] = [w / 2, h / 2]
    kp_lm = np.where(np.arange(nkps) < nobs_mp, np.arange(nkps), -1).astype(np.int32)
    order = rng.permutation(nkps)
    kp_px, kp_lm_src = kp_px[order], kp_lm[order]
    # map point table: [observed map points | candidates]
    nm = nobs_mp + ncand
    xyz = np.zeros((nm, 3))
    xyz[:nobs_mp] = world[:nobs_mp]
    base_desc = rng.integers(0, 256, (nm, 32), dtype=np.uint8)
    dup = rng.random(ncand) < 0.5
    src = rng.integers(0, nobs_mp, ncand)
    for c in range(ncand):
        m = nobs_mp + c
        if dup[c]:
            xyz[m] = xyz[src[c]] + rng.normal(0, 0.01, 3)
            d = base_desc[src[c]].copy()
            for b in rng.integers(0, 256, rng.integers(0, 30)):
                d[b >> 3] ^= np.uint8(1 << (b & 7))
            base_desc[m] = d
        else:
            zz = rng.uniform(1.0, 12.0)
            p = np.array([(rng.uniform(-60, w + 60) - K[2]) / K[0] * zz, (rng.uniform(-60, h + 60) - K[3]) / K[1] * zz, zz])
            if rng.random() < 0.05:
                p[2] = -p[2]
            xyz[m] = (p - t) @ R
    desc_ptr, descs = [0], []
    for m in range(nm):
        nd = int(rng.integers(1, 5)) if rng.random() > 0.03 else 0     # a few map points without descriptor
        for _ in range(nd):
            d = base_desc[m].copy()
            for b in rng.integers(0, 256, rng.integers(0, 6)):
                d[b >> 3] ^= np.uint8(1 << (b & 7))
            descs.append(d)
        desc_ptr.append(len(descs))
    kfmask = np.zeros((nm, 4), np.uint64)
    obs_ptr, obs_kf, obs_px = [0], [], []
    for m in range(nm):
        if m >= nobs_mp and dup[m - nobs_mp] and rng.random() < 0.8:
            free = [k for k in range(nkfs) if not (int(kfmask[src[m - nobs_mp], k >> 6]) >> (k & 63)) & 1]
            kfs = rng.choice(free, min(len(free), int(rng.integers(1, 4))), replace=False) if free else []
        else:
            kfs = rng.choice(nkfs, int(rng.integers(1, 6)), replace=False)
        for k in sorted(int(v) for v in kfs):
            kfmask[m, k >> 6] |= np.uint64(1) << np.uint64(k & 63)
            T = kf_T[k]
            cp = T[:9].reshape(3, 3) @ xyz[m] + T[9:]
            if cp[2] < 0.2:
                cp[2] = 0.2
            q = _proj_radtan(cp[None], K, dist)[0] + rng.normal(0, 0.7, 2)
            obs_kf.append(k)
            obs_px.append(q)
        obs_ptr.append(len(obs_kf))
    nbw, nbh = int(np.ceil(np.float32(w) / ncellsize)), int(np.ceil(np.float32(h) / ncellsize))
    cell = (np.floor(kp_px[:, 1] / np.float32(ncellsize)).astype(int) * nbw + np.floor(kp_px[:, 0] / np.float32(ncellsize)).astype(int))
    cell_kp = np.argsort(cell, kind="stable").astype(np.int32)
    cell_ptr = np.concatenate([[0], np.cumsum(np.bincount(cell, minlength=nbw * nbh))]).astype(np.int32)
    vfov, hfov = 0.5 * h / K[1], 0.5 * w / K[0]
    view_th = np.float32(np.cos(np.float32(np.arctan(np.float32(max(vfov, hfov))))))
    return dict(K=K, dist=dist, img_w=w, img_h=h, ncellsize=ncellsize, nbwcells=nbw, Tcw=Tcw, cell_ptr=cell_ptr, cell_kp=cell_kp,
                kp_px=np.ascontiguousarray(kp_px, np.float32), kp_lm=np.ascontiguousarray(kp_lm_src, np.int32),
                mp_xyz=xyz, mp_desc_ptr=np.asarray(desc_ptr, np.int32),
                desc=np.asarray(descs, np.uint8).reshape(-1, 32), mp_kfmask=kfmask,
                mp_obs_ptr=np.asarray(obs_ptr, np.int32), obs_kf=np.asarray(obs_kf, np.int32),
                obs_px=np.asarray(obs_px, np.float32).reshape(-1, 2), kf_Tcw=kf_T,
                cand_mp=(nobs_mp + rng.permutation(ncand)).astype(np.int32),
                dmaxpxdist=np.float32(2.0 * 2), fdistratio=np.float32(0.2), view_th=view_th)
