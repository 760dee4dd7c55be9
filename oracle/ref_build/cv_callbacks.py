"""The real OpenCV (cv2) behind the stand-in OpenCV containers of oracle/ref_build/mini_cv: every arithmetic call the reference's
feature extractor makes is answered here by the cv2 function of the same name, on views of the C++ side's buffers.
TEST INFRASTRUCTURE: only tests/ use this."""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from pathlib import Path

import cv2
import numpy as np

HERE = Path(__file__).resolve().parent
OUT = HERE.parent / "_ref" / "libov2ref_frontend.so"
REF = Path("/root/reference")
SRC = REF / "src" / "feature_extractor.cpp"
SRC2 = REF / "src" / "feature_tracker.cpp"

U8P, F32P, F64P, I32P = C.POINTER(C.c_uint8), C.POINTER(C.c_float), C.POINTER(C.c_double), C.POINTER(C.c_int)
_DT = {0: np.uint8, 5: np.float32, 6: np.float64}


def _view(ptr, rows, cols, step, dtype):
    """numpy view (rows, cols) of a C buffer with a row step in bytes (ROIs share their parent's step)."""
    dt = np.dtype(dtype)
    buf = (C.c_uint8 * (step * (rows - 1) + cols * dt.itemsize)).from_address(C.addressof(ptr.contents))
    return np.ndarray((rows, cols), dt, buf, 0, (step, dt.itemsize))


@C.CFUNCTYPE(None, U8P, C.c_int, C.c_int, C.c_size_t, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, C.c_int)
def _circle(data, rows, cols, step, typ, cx, cy, radius, color, thickness):
    cv2.circle(_view(data, rows, cols, step, _DT[typ]), (cx, cy), radius, color, thickness)


@C.CFUNCTYPE(C.c_int, C.c_int, U8P, C.c_int, C.c_int, C.c_size_t, U8P, C.c_size_t, C.c_int, F32P, C.c_int)
def _fast_detect(th, img, rows, cols, step, mask, mask_step, mask_type, out, cap):
    roi = _view(img, rows, cols, step, np.uint8)
    m = _view(mask, rows, cols, mask_step, _DT[mask_type]) if mask else None
    kps = cv2.FastFeatureDetector_create(int(th)).detect(roi, m)
    n = min(len(kps), cap)
    for i in range(n):
        out[3 * i], out[3 * i + 1], out[3 * i + 2] = kps[i].pt[0], kps[i].pt[1], kps[i].response
    return n


@C.CFUNCTYPE(None, U8P, C.c_int, C.c_int, C.c_size_t, F32P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double)
def _corner_subpix(img, rows, cols, step, pts, n, win, zero, max_iter, eps):
    im = _view(img, rows, cols, step, np.uint8)
    p = np.ctypeslib.as_array(pts, (n, 2))
    q = np.ascontiguousarray(p.reshape(n, 1, 2), np.float32)
    cv2.cornerSubPix(im, q, (win, win), (zero, zero), (cv2.TERM_CRITERIA_EPS + cv2.TERM_CRITERIA_MAX_ITER, max_iter, eps))
    p[...] = q.reshape(n, 2)


@C.CFUNCTYPE(None, U8P, C.c_int, C.c_int, C.c_size_t, C.c_int, C.c_int, C.c_int, C.c_int, U8P, C.c_int, C.c_double)
def _gaussian_blur(parent, prows, pcols, step, px, py, rows, cols, out, ksize, sigma):
    """cv::GaussianBlur.  On a ROI the C++ library filters with the PARENT's pixels beyond the ROI's edge (it knows the parent through
    datastart / dataend); a numpy slice handed to cv2 loses that, so the ROI case is composed from whole-image cv2 calls by
    oracle/image_ref.py::blur3_cell_cv2 (the 3 x 3, sigma 0, square-cell case the reference uses)."""
    from oracle import image_ref as R
    im = _view(parent, prows, pcols, step, np.uint8)
    o = np.ctypeslib.as_array(out, (rows, cols))
    if px == 0 and py == 0 and rows == prows and cols == pcols:
        o[...] = cv2.GaussianBlur(im, (ksize, ksize), sigma)
    else:
        assert ksize == 3 and sigma == 0 and rows == cols
        o[...] = R.blur3_cell_cv2(np.ascontiguousarray(im), px, py, rows)


@C.CFUNCTYPE(None, U8P, C.c_int, C.c_int, C.c_size_t, F32P, C.c_int, C.c_int)
def _corner_min_eigen(img, rows, cols, step, out, block, ksize):
    o = np.ctypeslib.as_array(out, (rows, cols))
    o[...] = cv2.cornerMinEigenVal(_view(img, rows, cols, step, np.uint8), block, ksize=ksize)


@C.CFUNCTYPE(None, F32P, C.c_int, C.c_int, C.c_size_t, F64P, F64P, I32P, I32P)
def _min_max_loc(m, rows, cols, step, minv, maxv, minxy, maxxy):
    a = _view(C.cast(m, U8P), rows, cols, step, np.float32)
    lo, hi, plo, phi = cv2.minMaxLoc(a)
    minv[0], maxv[0] = lo, hi
    minxy[0], minxy[1], maxxy[0], maxxy[1] = plo[0], plo[1], phi[0], phi[1]


_ORB = None


@C.CFUNCTYPE(C.c_int, U8P, C.c_int, C.c_int, C.c_size_t, F32P, C.c_int, U8P)
def _orb_compute(img, rows, cols, step, pts, n, desc_out):
    global _ORB
    if _ORB is None:
        _ORB = cv2.ORB_create(500, 1.0, 0)
    im = _view(img, rows, cols, step, np.uint8)
    p = np.ctypeslib.as_array(pts, (n, 2))
    kps = [cv2.KeyPoint(float(x), float(y), 1.0) for x, y in p]          # KeyPoint::convert: size 1, angle -1, octave 0
    kps, desc = _ORB.compute(np.ascontiguousarray(im), kps)
    m = len(kps)
    for i in range(m):
        p[i, 0], p[i, 1] = kps[i].pt
    if m:
        np.ctypeslib.as_array(desc_out, (m, 32))[...] = desc
    return m


@C.CFUNCTYPE(None, U8P, U8P, C.c_int, C.c_int, C.c_size_t, C.c_size_t, F32P, F32P, C.c_int, U8P, F32P, C.c_int, C.c_int, C.c_int, C.c_double, C.c_int, C.c_double)
def _lk(prev, nxt, rows, cols, pstep, nstep, prev_pts, next_pts, n, status, err, win, max_level, max_iter, eps, flags, min_eig):
    a, b = _view(prev, rows, cols, pstep, np.uint8), _view(nxt, rows, cols, nstep, np.uint8)
    p0 = np.ascontiguousarray(np.ctypeslib.as_array(prev_pts, (n, 2)), np.float32).reshape(n, 1, 2)
    nx = np.ctypeslib.as_array(next_pts, (n, 2))
    p1 = np.ascontiguousarray(nx, np.float32).reshape(n, 1, 2).copy()
    p1, st, er = cv2.calcOpticalFlowPyrLK(np.ascontiguousarray(a), np.ascontiguousarray(b), p0, p1, winSize=(win, win), maxLevel=max_level,
                                          criteria=(cv2.TERM_CRITERIA_COUNT + cv2.TERM_CRITERIA_EPS, max_iter, eps), flags=flags, minEigThreshold=min_eig)
    nx[...] = p1.reshape(n, 2)
    np.ctypeslib.as_array(status, (n,))[...] = st.reshape(n)
    np.ctypeslib.as_array(err, (n,))[...] = er.reshape(n)


@C.CFUNCTYPE(None, U8P, C.c_int, C.c_int, C.c_size_t, C.c_int, C.c_int, C.c_float, C.c_float, U8P)
def _get_rect_subpix(img, rows, cols, step, pw, ph, cx, cy, out):
    im = _view(img, rows, cols, step, np.uint8)
    np.ctypeslib.as_array(out, (ph, pw))[...] = cv2.getRectSubPix(np.ascontiguousarray(im), (pw, ph), (cx, cy))


class _Callbacks(C.Structure):
    _fields_ = [("circle", C.c_void_p), ("fast_detect", C.c_void_p), ("corner_subpix", C.c_void_p), ("gaussian_blur", C.c_void_p),
                ("corner_min_eigen", C.c_void_p), ("min_max_loc", C.c_void_p), ("orb_compute", C.c_void_p), ("lk", C.c_void_p), ("get_rect_subpix", C.c_void_p)]


_KEEP = (_circle, _fast_detect, _corner_subpix, _gaussian_blur, _corner_min_eigen, _min_max_loc, _orb_compute, _lk, _get_rect_subpix)


def available() -> bool:
    return OUT.exists() or SRC.exists()


def build(force: bool = False):
    """oracle/_ref/libov2ref_frontend.so: the reference's src/feature_extractor.cpp and src/feature_tracker.cpp (in place) + fe_ref.cpp, against mini_cv (OpenCV
    containers), the reference tree's Sophus and the stand-in Eigen header."""
    if not os.access(SRC, os.R_OK):
        return OUT if OUT.exists() else None
    deps = [SRC, SRC2, HERE / "fe_ref.cpp"] + [p for d in ("mini", "mini_cv") for p in (HERE / d).rglob("*") if p.is_file()]
    if not force and OUT.exists() and all(OUT.stat().st_mtime >= d.stat().st_mtime for d in deps):
        return OUT
    OUT.parent.mkdir(parents=True, exist_ok=True)
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-w", "-I", str(HERE / "mini_cv"), "-I", str(REF / "Thirdparty" / "Sophus"),
                           "-I", str(HERE / "mini"), "-I", str(REF / "include"), str(SRC), str(SRC2), str(HERE / "fe_ref.cpp"), "-o", str(OUT)])
    return OUT


def load():
    """The library with the cv2 callbacks installed, or None when it cannot be built here."""
    so = build()
    if so is None:
        return None
    lib = C.CDLL(str(so))
    cb = _Callbacks(*[C.cast(f, C.c_void_p) for f in _KEEP])
    lib.ov2ref_cv_set_callbacks(C.byref(cb))
    lib.ov2ref_fe_create.restype = C.c_void_p
    lib.ov2ref_fe_create.argtypes = [C.c_int, C.c_int, C.c_double, C.c_int]
    lib.ov2ref_fe_destroy.argtypes = [C.c_void_p]
    for name in ("ov2ref_fe_detect_grid_fast", "ov2ref_fe_detect_single_scale", "ov2ref_fe_describe", "ov2ref_ft_fb_klt"):
        getattr(lib, name).restype = C.c_int
    return lib
