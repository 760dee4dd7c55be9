"""The restatements (oracle/ba_ref.py, oracle/pnp_ref.py) against the REFERENCE'S OWN residual source: oracle/_ref/libov2ref_residuals.so
is /root/reference/src/ceres_parametrization.cpp compiled where it lies (recipe oracle/ref_build/build_ref.py) with the reference tree's own
Sophus 1.1 and Ceres 2.0 public headers, against a stand-in Eigen header (oracle/ref_build/mini: this container has no Eigen).  Pins rows R and Q of the scope table
(residuals, chi2 / depth flags, every Jacobian block, SE3LeftParameterization::Plus) and the ceresPnP residual to what the
reference's code computes."""
import ctypes as C

import numpy as np
import pytest

from oracle import ba_ref as B
from oracle import pnp_ref as P
from oracle.ref_build import build_ref
from reference_calls import library

K = np.array([458.654, 457.296, 367.215, 248.375])
KR = np.array([457.587, 456.134, 379.999, 255.238])
D = C.POINTER(C.c_double)


@pytest.fixture(scope="module")
def ref():
    def load():
        so = build_ref.build()
        return None if so is None else C.CDLL(str(so))
    with library("residuals", load) as lib:
        for name in ("ref_eval_anch_invdepth", "ref_eval_right_anch", "ref_eval_right_cam", "ref_eval_pnp", "ref_se3_plus"):
            getattr(lib, name).restype = C.c_int
        yield lib


def p(a):
    return a.ctypes.data_as(D)


def rand_pose(rng, scale=1.0, unit=True):
    q = rng.normal(0, 1, 4)
    q /= np.linalg.norm(q)
    if not unit:
        q *= rng.uniform(0.5, 2.0)                 # Sophus::SE3d(q, t) normalises (se3_param_block / Evaluate)
    return np.concatenate([rng.normal(0, scale, 3), q])


def scene(rng):
    """An anchor keyframe, an observer, a landmark seen by both with positive depth most of the time, and a stereo extrinsic."""
    Ta = rand_pose(rng, 0.5)
    Ta[3:] = B.quat_normalize(np.array([0.02, -0.03, 0.01, 1.0]) + rng.normal(0, 0.05, 4))
    To = Ta.copy()
    To[:3] += rng.normal(0, 0.3, 3)
    To[3:] = B.quat_normalize(To[3:] + rng.normal(0, 0.05, 4))
    Trl = np.concatenate([[-0.11, 0.001, 0.002] + rng.normal(0, 0.002, 3), B.quat_normalize(np.array([0.002, -0.003, 0.001, 1.0]))])
    invd = float(rng.uniform(0.08, 1.5)) * (1 if rng.random() > 0.1 else -1)      # a few points behind the camera
    ua = np.array([rng.uniform(20, 730), rng.uniform(20, 460)])
    u = np.array([rng.uniform(0, 752), rng.uniform(0, 480)])
    return Ta, To, Trl, invd, ua, u


def oracle_block(Ta, To, Trl, invd, ua, u, typ):
    pb = dict(K=K, Kr=KR, Trl=Trl, obs_lm=np.array([0]), lm_anchor_cam=np.array([0]), obs_cam=np.array([1]),
              lm_anchor_px=ua[None], obs_px=u[None], obs_type=np.array([typ], np.uint8))
    return B.evaluate(pb, np.stack([Ta, To]), np.array([invd]), np.array([0]))


def close(a, b):
    return np.allclose(a, b, rtol=1e-10, atol=1e-9)      # observed: 1.3e-13 relative over 2 000 random blocks


def test_mono_block_equals_the_reference_source(ref):
    """DirectLeftSE3::ReprojectionErrorKSE3AnchInvDepth::Evaluate (ceres_parametrization.cpp:361-473)."""
    rng = np.random.default_rng(1)
    nneg = 0
    for _ in range(300):
        Ta, To, Trl, invd, ua, u = scene(rng)
        res, Jk, Ja, Jo, Jl = np.zeros(2), np.ones(8), np.zeros(14), np.zeros(14), np.zeros(2)
        chi2, dpos = C.c_double(), C.c_int()
        assert ref.ref_eval_anch_invdepth(p(K), p(Ta), p(To), C.c_double(invd), C.c_double(u[0]), C.c_double(u[1]), C.c_double(ua[0]),
                                          C.c_double(ua[1]), C.c_double(1.0), p(res), p(Jk), p(Ja), p(Jo), p(Jl), C.byref(chi2), C.byref(dpos))
        o = oracle_block(Ta, To, Trl, invd, ua, u, 0)
        assert close(res, o["r"][0]) and close(chi2.value, o["chi2"][0]) and bool(dpos.value) == bool(o["depth_pos"][0])
        Ja, Jo = Ja.reshape(2, 7), Jo.reshape(2, 7)
        assert close(Ja[:, :6], o["Ja"][0]) and close(Jo[:, :6], o["Jo"][0]) and close(Jl, o["Jl"][0])
        assert not Ja[:, 6].any() and not Jo[:, 6].any() and not Jk.any()       # 7th column: the local parameterisation's zero row; K constant
        nneg += not dpos.value
    assert 5 < nneg < 100


def test_right_camera_blocks_equal_the_reference_source(ref):
    """...RightAnchCam... (:476-577) and ...RightCam... (:579-712)."""
    rng = np.random.default_rng(2)
    for _ in range(300):
        Ta, To, Trl, invd, ua, u = scene(rng)
        res, Jkl, Jkr, Jrl, Jl = np.zeros(2), np.ones(8), np.ones(8), np.ones(14), np.zeros(2)
        chi2, dpos = C.c_double(), C.c_int()
        assert ref.ref_eval_right_anch(p(K), p(KR), p(Trl), C.c_double(invd), C.c_double(u[0]), C.c_double(u[1]), C.c_double(ua[0]),
                                       C.c_double(ua[1]), C.c_double(1.0), p(res), p(Jkl), p(Jkr), p(Jrl), p(Jl), C.byref(chi2), C.byref(dpos))
        o = oracle_block(Ta, To, Trl, invd, ua, u, 2)
        assert close(res, o["r"][0]) and close(chi2.value, o["chi2"][0]) and bool(dpos.value) == bool(o["depth_pos"][0])
        assert close(Jl, o["Jl"][0]) and not o["Ja"].any() and not o["Jo"].any()
        # (the calibration / extrinsic Jacobians the reference fills here are never used: localBA holds those blocks constant,
        #  optimizer.cpp:98,113,125)
        res, Ja, Jo = np.zeros(2), np.zeros(14), np.zeros(14)
        Jkl, Jkr, Jrl = np.ones(8), np.ones(8), np.ones(14)
        assert ref.ref_eval_right_cam(p(K), p(KR), p(Ta), p(To), p(Trl), C.c_double(invd), C.c_double(u[0]), C.c_double(u[1]), C.c_double(ua[0]),
                                      C.c_double(ua[1]), C.c_double(1.0), p(res), p(Jkl), p(Jkr), p(Ja), p(Jo), p(Jrl), p(Jl), C.byref(chi2),
                                      C.byref(dpos))
        o = oracle_block(Ta, To, Trl, invd, ua, u, 1)
        assert close(res, o["r"][0]) and close(chi2.value, o["chi2"][0]) and bool(dpos.value) == bool(o["depth_pos"][0])
        Ja, Jo = Ja.reshape(2, 7), Jo.reshape(2, 7)
        assert close(Ja[:, :6], o["Ja"][0]) and close(Jo[:, :6], o["Jo"][0]) and close(Jl, o["Jl"][0])
        assert not Ja[:, 6].any() and not Jo[:, 6].any()


def test_pnp_block_equals_the_reference_source(ref):
    """DirectLeftSE3::ReprojectionErrorSE3::Evaluate (:301-358), with the per-octave sigma = 2^scale the front-end passes."""
    rng = np.random.default_rng(3)
    for _ in range(300):
        T = rand_pose(rng, 1.0, unit=rng.random() > 0.3)
        w = rng.normal(0, 3, 3)
        u = np.array([rng.uniform(0, 752), rng.uniform(0, 480)])
        scale = int(rng.integers(0, 3))
        res, J = np.zeros(2), np.zeros(14)
        chi2, dpos = C.c_double(), C.c_int()
        assert ref.ref_eval_pnp(p(K), p(T), p(w), C.c_double(u[0]), C.c_double(u[1]), C.c_double(2.0 ** scale), p(res), p(J), C.byref(chi2), C.byref(dpos))
        o = P.evaluate(T, w[None], u[None], K, scales=[scale])
        J = J.reshape(2, 7)
        assert close(res, o["r"][0]) and close(chi2.value, o["chi2"][0]) and bool(dpos.value) == bool(o["depth_pos"][0])
        assert close(J[:, :6], o["J"][0]) and not J[:, 6].any()


def test_se3_left_plus_equals_the_reference_source(ref):
    """SE3LeftParameterization::Plus (se3left_parametrization.hpp:41-60): exp(delta) * T, small-angle branch included; its 7 x 6
    Jacobian is [I; 0], which is why only the first six columns of the 2 x 7 blocks above matter."""
    rng = np.random.default_rng(4)
    for k in range(400):
        T = rand_pose(rng, 2.0, unit=rng.random() > 0.3)
        mag = [1e-13, 1e-11, 1e-9, 1e-6, 1e-3, 0.1, 1.0, 3.0][k % 8]
        delta = np.concatenate([rng.normal(0, 0.5, 3), rng.normal(0, 1, 3) * mag])
        out, J = np.zeros(7), np.zeros(42)
        assert ref.ref_se3_plus(p(T), p(delta), p(out), p(J))
        want = B.pose_plus(T, delta)
        assert close(out, want)
        assert np.array_equal(J.reshape(7, 6), np.vstack([np.eye(6), np.zeros((1, 6))]))
