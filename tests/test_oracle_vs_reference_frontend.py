"""oracle/image_ref.py's restatement of the reference's feature extractor against the REFERENCE'S OWN SOURCE: oracle/_ref/libov2ref_frontend.so
is /root/reference/src/feature_extractor.cpp compiled where it lies against stand-in OpenCV containers whose arithmetic calls (FAST,
cornerSubPix, GaussianBlur, cornerMinEigenVal, minMaxLoc, circle, ORB::compute) are answered by the real OpenCV through callbacks
(oracle/ref_build/mini_cv, cv_callbacks.py).  So the reference's control flow - grid walk in ascending cell order, the float mask and
its discs, libstdc++'s std::sort on the FAST responses, threshold / quality adaptation across frames, second detections, the
descriptor re-alignment - runs as written, on the real library's numbers; the numpy restatement (the non-cv2 code path, which is what
the CUDA kernels are compared with) must give the same keypoints, thresholds and descriptors."""
import ctypes as C

import numpy as np
import pytest

from oracle import image_ref as R
from ov2slam_b200 import synth
from reference_calls import library

cv2 = pytest.importorskip("cv2")


@pytest.fixture(scope="module")
def ref():
    from oracle.ref_build import cv_callbacks as CB
    with library("frontend", CB.load) as lib:
        yield lib, CB


def _call(ref, name, fe, im, cs, cur, roi, state_type):
    lib, CB = ref
    out = np.zeros((8192, 2), np.float32)
    state = state_type()
    cur = np.ascontiguousarray(cur, np.float32).reshape(-1, 2)
    roi = np.asarray(roi, np.int32)
    im = np.ascontiguousarray(im)
    n = getattr(lib, name)(C.c_void_p(fe), im.ctypes.data_as(CB.U8P), im.shape[0], im.shape[1], cs, cur.ctypes.data_as(CB.F32P), len(cur),
                           roi.ctypes.data_as(CB.I32P), out.ctypes.data_as(CB.F32P), len(out), C.byref(state))
    return out[:n].copy(), state.value


@pytest.mark.parametrize("w,h,cs", [(640, 480, 50), (752, 480, 35), (333, 245, 16)])
def test_detect_grid_fast_equals_the_reference_source(ref, w, h, cs, capfd):
    """Three frames through ONE extractor (the adaptive threshold carries over), the second and third with the tracked keypoints of the
    frame before as existing keypoints."""
    lib, _ = ref
    fe = lib.ov2ref_fe_create(1000, 50, 0.001, 10)
    th = 10
    cur = np.zeros((0, 2), np.float32)
    seen_th = set()
    for k in range(3):
        im = synth.make_pair(40 + k, w, h)[0]
        got, got_th = _call(ref, "ov2ref_fe_detect_grid_fast", fe, im, cs, cur, (5, 5, w - 10, h - 10), C.c_int)
        ipts, want_th, _ = R.detect_grid_fast_nosubpix(im, cs, cur, th, use_cv2=False)
        want = R.corner_subpix_cv2(im, ipts.astype(np.float32)) if len(ipts) else np.zeros((0, 2), np.float32)
        assert got_th == want_th and len(got) == len(want) > 10
        assert np.array_equal(got, want)
        th = want_th
        seen_th.add(th)
        cur = got[::3] + np.float32(0.37)                       # some of them "tracked" into the next frame, off the pixel grid
    lib.ov2ref_fe_destroy(C.c_void_p(fe))


def test_fast_threshold_adaptation_equals_the_reference_source(ref):
    """A bland image (few corners: threshold * 0.66 per frame, 10 -> 6 -> 3 -> 1 -> 0) and a corner in every cell (threshold * 1.5)."""
    lib, _ = ref
    rng = np.random.default_rng(3)
    bland = (128 + 3 * rng.standard_normal((240, 320))).clip(0, 255).astype(np.uint8)
    fe = lib.ov2ref_fe_create(1000, 50, 0.001, 10)
    th, ths = 10, []
    for _ in range(5):
        got, got_th = _call(ref, "ov2ref_fe_detect_grid_fast", fe, bland, 50, np.zeros((0, 2)), (0, 0, 320, 240), C.c_int)
        ipts, th, _ = R.detect_grid_fast_nosubpix(bland, 50, np.zeros((0, 2)), th, use_cv2=False)
        assert got_th == th and len(got) == len(ipts)
        ths.append(th)
    assert ths[:4] == [6, 3, 1, 0]
    lib.ov2ref_fe_destroy(C.c_void_p(fe))
    busy = synth.make_pair(9, 320, 240)[0]
    fe = lib.ov2ref_fe_create(1000, 50, 0.001, 4)
    got, got_th = _call(ref, "ov2ref_fe_detect_grid_fast", fe, busy, 50, np.zeros((0, 2)), (0, 0, 320, 240), C.c_int)
    ipts, th, nbempty = R.detect_grid_fast_nosubpix(busy, 50, np.zeros((0, 2)), 4, use_cv2=False)
    assert got_th == th and len(got) == len(ipts)
    lib.ov2ref_fe_destroy(C.c_void_p(fe))


@pytest.mark.parametrize("w,h,cs", [(640, 480, 50), (752, 480, 35), (1280, 720, 35)])
def test_detect_single_scale_equals_the_reference_source(ref, w, h, cs):
    """Two frames through one extractor (dmaxquality_ adapts), the second with existing keypoints and a roi that cuts cells off."""
    lib, _ = ref
    fe = lib.ov2ref_fe_create(1000, 50, 0.001, 10)
    q = 0.001
    cur = np.zeros((0, 2), np.float32)
    for k, roi in enumerate(((5, 5, w - 10, h - 10), (40, 30, w - 120, h - 90))):
        im = synth.make_pair(50 + k, w, h)[0]
        got, got_q = _call(ref, "ov2ref_fe_detect_single_scale", fe, im, cs, cur, roi, C.c_double)
        ipts, want_q, _ = R.detect_single_scale_nosubpix(im, cs, cur, roi, q, use_cv2=False)
        want = R.corner_subpix_cv2(im, ipts.astype(np.float32)) if len(ipts) else np.zeros((0, 2), np.float32)
        assert got_q == want_q and len(got) == len(want) > 10
        assert np.array_equal(got, want)
        q = want_q
        cur = got[::2] + np.float32(0.25)
    lib.ov2ref_fe_destroy(C.c_void_p(fe))


@pytest.mark.parametrize("w,h", [(640, 480), (333, 245)])
def test_describe_brief_equals_the_reference_source(ref, w, h):
    """describeBRIEF's non-contrib branch (cv::ORB::create(500, 1., 0)): points near the border get an empty Mat, the rest are
    re-aligned by exact pixel equality; descriptors of the numpy restatement equal the reference's, bit for bit."""
    lib, CB = ref
    im = synth.make_pair(60, w, h)[0]
    rng = np.random.default_rng(6)
    pts = np.stack([rng.uniform(0, w, 400), rng.uniform(0, h, 400)], 1).astype(np.float32)
    pts[:5] = [[31, 31], [30.9, 40], [w - 32, h - 32], [w - 31, 50], [100.5, 30.99]]
    fe = lib.ov2ref_fe_create(1000, 50, 0.001, 10)
    desc, valid = np.zeros((len(pts), 32), np.uint8), np.zeros(len(pts), np.uint8)
    n = lib.ov2ref_fe_describe(C.c_void_p(fe), im.ctypes.data_as(CB.U8P), h, w, pts.ctypes.data_as(CB.F32P), len(pts), desc.ctypes.data_as(CB.U8P),
                               valid.ctypes.data_as(CB.U8P))
    assert n == len(pts)
    rd, rv = R.describe_ref(im, pts)
    assert np.array_equal(valid, rv) and 0.5 < valid.mean() < 1.0
    assert np.array_equal(desc[valid > 0], rd[rv > 0])
    lib.ov2ref_fe_destroy(C.c_void_p(fe))


@pytest.mark.parametrize("w,h,nbpyrlvl,npyr_entries", [(640, 480, 3, 8), (640, 480, 1, 8), (752, 480, 3, 4)])
def test_fb_klt_tracking_equals_the_reference_source(ref, w, h, nbpyrlvl, npyr_entries):
    """FeatureTracker::fbKltTracking as written (/root/reference/src/feature_tracker.cpp:35-137: level clamp against the pyramid's size,
    forward track from the priors, error / border tests, backward track on level 0, forward-backward distance) on the real library's
    Lucas-Kanade, against the oracle's orchestration around the same cv2 call; and the exact-integer restatement the kernels are compared
    with gives the same statuses."""
    lib, CB = ref
    prev, cur, flow = synth.make_pair(70, w, h)
    rng = np.random.default_rng(7)
    n = 400
    kps = np.stack([rng.uniform(0, w, n), rng.uniform(0, h, n)], 1).astype(np.float32)
    kps[:6] = [[0.5, 0.5], [w - 1.2, h - 1.2], [3, h / 2], [w / 2, 2], [w - 3, 10], [20, h - 2.5]]      # border points
    pri = (kps + np.asarray(flow, np.float32) + rng.normal(0, 1.5, (n, 2))).astype(np.float32)
    got_pri, st = pri.copy(), np.zeros(n, np.uint8)
    m = lib.ov2ref_ft_fb_klt(prev.ctypes.data_as(CB.U8P), cur.ctypes.data_as(CB.U8P), h, w, npyr_entries, 9, nbpyrlvl, C.c_float(30.0), C.c_float(0.5), 30,
                             C.c_float(0.01), kps.ctypes.data_as(CB.F32P), got_pri.ctypes.data_as(CB.F32P), n, st.ctypes.data_as(CB.U8P))
    assert m == n
    eff = min(nbpyrlvl, npyr_entries // 2 - 1)                # the clamp (:50-52)
    want_pri, want_st = R._fb_klt(R._lk_cv2, prev, cur, kps, pri, 9, eff, 30.0, 0.5, 30, R.KLT_EPS)
    assert np.array_equal(st, want_st) and 0.3 < st.mean() < 1.0
    assert np.array_equal(got_pri, want_pri)
    ref_pri, ref_st = R._fb_klt(R._lk_ref, prev, cur, kps, pri, 9, eff, 30.0, 0.5, 30, R.KLT_EPS)
    assert (ref_st != st).mean() <= 0.01                      # cv2's float SIMD lane order vs exact sums: a borderline track may flip
    both = (ref_st > 0) & (st > 0)
    assert np.abs(ref_pri[both] - got_pri[both]).max() <= 1e-2


def test_get_line_min_sad_equals_the_reference_source(ref):
    """FeatureTracker::getLineMinSAD as written (:138-204) on the real library's getRectSubPix, against the restatement (window rule
    incl. the growing window at the right / bottom edge, sub-pixel patches, scan direction, strict minimum).  cv2 builds with Intel IPP
    sample sub-pixel patches one grey level differently on ~0.7 % of the pixels: the column may then differ on a near-tie."""
    lib, CB = ref
    left = synth.make_pair(80, 160, 120)[0]
    right = np.roll(left, -6, axis=1)
    rng = np.random.default_rng(8)
    nsame = ntot = 0
    for k in range(120):
        x, y = float(np.float32(rng.uniform(0, 160))), float(np.float32(rng.uniform(0, 120)))
        if k < 8:
            x, y = [(1.2, 40.0), (158.7, 60.0), (80.0, 1.4), (80.0, 118.8), (159.4, 119.4), (0.3, 0.3), (3.0, 3.0), (156.5, 3.2)][k]
        for goleft in (1, 0):
            xp, er = C.c_float(-7), C.c_float(-7)
            lib.ov2ref_ft_line_min_sad(left.ctypes.data_as(CB.U8P), right.ctypes.data_as(CB.U8P), 120, 160, C.c_float(x), C.c_float(y), 7, goleft,
                                       C.byref(xp), C.byref(er))
            wx, we = R.line_min_sad_ref(left, right, (x, y), 7, bool(goleft))
            ntot += 1
            if xp.value == wx:
                nsame += 1
                assert wx < 0 or abs(er.value - we) <= 0.5          # mean absolute difference over 49 pixels, a few of them one grey level off
    assert nsame >= 0.97 * ntot
