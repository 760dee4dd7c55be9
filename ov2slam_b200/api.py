"""ctypes binding of libov2b200.so (include/ov2b200.h) + thin numpy/torch-friendly wrappers.

This is the Python-side mirror of the reference's operator interface for the hot paths:

    FeatureTracker.fb_klt_tracking   <- FeatureTracker::fbKltTracking   (feature_tracker.cpp:35-137)
    FeatureExtractor.detect_grid_fast<- FeatureExtractor::detectGridFAST(feature_extractor.cpp:443-570)
    FeatureExtractor.describe_brief  <- FeatureExtractor::describeBRIEF (feature_extractor.cpp:224-285)
    Optimizer.local_ba               <- Optimizer::localBA solve part   (optimizer.cpp:436-735)

Everything computes on the GPU through the C ABI.  There is NO CPU fallback: if the shared
library is missing it is an ImportError-like failure (Ov2Error), if no CUDA device is present
ov2_create() returns OV2_ERR_NO_DEVICE.  Nothing here imports oracle/.
"""
from __future__ import annotations

import ctypes as C
import weakref
from pathlib import Path

import numpy as np

_LIBPATH = Path(__file__).resolve().parent / "lib" / "libov2b200.so"
_lib = None

OV2_OK = 0
STATUS_NAMES = {0: "OK", 1: "NO_DEVICE", 2: "CUDA", 3: "INVALID", 4: "CAPACITY", 5: "NOMEM", 6: "NUMERIC"}

ABI_SYMBOLS = [
    "ov2_create", "ov2_destroy", "ov2_last_error", "ov2_version", "ov2_set_stream", "ov2_sync",
    "ov2_batch_begin", "ov2_batch_end",
    "ov2_host_alloc", "ov2_host_free", "ov2_launch_count", "ov2_profile_enable", "ov2_profile_query",
    "ov2_pyr_create", "ov2_pyr_destroy", "ov2_pyr_build", "ov2_pyr_download", "ov2_clahe", "ov2_preprocess",
    "ov2_fb_klt", "ov2_grid_fast", "ov2_detect_single_scale", "ov2_pnp_solve", "ov2_debug_fast_cells", "ov2_describe", "ov2_describe_config", "ov2_line_min_sad", "ov2_match_to_map", "ov2_frontend_step", "ov2_localba_solve", "ov2_localba_solve_sharded", "ov2_localba_solve_batch", "ov2_localba_request_stop",
    "ov2_ba_comm_create", "ov2_ba_comm_handle", "ov2_ba_comm_connect", "ov2_ba_comm_connect_local", "ov2_ba_comm_destroy", "ov2_localba_solve_p2p",
]


class Ov2Error(RuntimeError):
    pass


class KltParams(C.Structure):
    _fields_ = [("win", C.c_int), ("max_iter", C.c_int), ("eps", C.c_float), ("ferr", C.c_float),
                ("fb_dist", C.c_float)]


class FrontendStepArgs(C.Structure):
    _fields_ = [("prev_images", C.c_void_p), ("cur_images", C.c_void_p), ("row_stride", C.c_size_t), ("frame_stride", C.c_size_t),
                ("count", C.c_int), ("klt", KltParams), ("n_kps", C.c_int), ("kps_per_frame", C.c_int),
                ("nbpyrlvl", C.c_void_p), ("nbpyrlvl_all", C.c_int), ("kps", C.c_void_p), ("priors_inout", C.c_void_p),
                ("status_out", C.c_void_p), ("cellsize", C.c_int), ("fast_th_inout", C.c_void_p), ("max_per_frame", C.c_int),
                ("new_pts", C.c_void_p), ("new_counts", C.c_void_p), ("desc_tracked", C.c_void_p), ("valid_tracked", C.c_void_p),
                ("desc_new", C.c_void_p), ("valid_new", C.c_void_p)]


class BaProblem(C.Structure):
    _fields_ = [("ncam", C.c_int32), ("npts", C.c_int32), ("nobs", C.c_int32),
                ("K", C.c_void_p), ("pose", C.c_void_p), ("pose_const", C.c_void_p),
                ("lm_anchor_cam", C.c_void_p), ("lm_anchor_px", C.c_void_p), ("lm_invdepth", C.c_void_p),
                ("obs_cam", C.c_void_p), ("obs_lm", C.c_void_p), ("obs_px", C.c_void_p),
                ("obs_type", C.c_void_p), ("Kr", C.c_void_p), ("Trl", C.c_void_p)]


class MatchProblem(C.Structure):
    """ov2_match_problem (include/ov2b200.h), field for field."""
    _fields_ = [("Tcw", C.c_double * 12), ("K", C.c_double * 4), ("dist", C.c_void_p),
                ("img_w", C.c_int), ("img_h", C.c_int), ("ncellsize", C.c_int), ("nbwcells", C.c_int), ("ncells", C.c_int),
                ("cell_ptr", C.c_void_p), ("cell_kp", C.c_void_p), ("nkps", C.c_int), ("kp_px", C.c_void_p), ("kp_lm", C.c_void_p),
                ("nmps", C.c_int), ("mp_xyz", C.c_void_p), ("mp_desc_ptr", C.c_void_p), ("ndesc", C.c_int), ("desc", C.c_void_p),
                ("mp_kfmask", C.c_void_p), ("mp_obs_ptr", C.c_void_p), ("nobs", C.c_int), ("obs_kf", C.c_void_p), ("obs_px", C.c_void_p),
                ("nkfs", C.c_int), ("kf_Tcw", C.c_void_p), ("ncand", C.c_int), ("cand_mp", C.c_void_p),
                ("dmaxpxdist", C.c_float), ("fdistratio", C.c_float), ("view_th", C.c_float)]


class BaOpts(C.Structure):
    _fields_ = [("max_iters_robust", C.c_int), ("max_iters_refine", C.c_int), ("huber_th", C.c_double),
                ("function_tolerance", C.c_double), ("use_robust", C.c_int), ("apply_l2_after_robust", C.c_int),
                ("refine_loss", C.c_int)]


class BaResult(C.Structure):
    _fields_ = [("iters_robust", C.c_int), ("iters_refine", C.c_int), ("initial_cost", C.c_double),
                ("final_cost", C.c_double), ("n_outliers_first", C.c_int), ("n_outliers_second", C.c_int),
                ("termination", C.c_int)]


ALLREDUCE_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p)


def lib_path() -> Path:
    return _LIBPATH


def load():
    """Load the shared library (build it first with ov2slam_b200.build.build())."""
    global _lib
    if _lib is not None:
        return _lib
    if not _LIBPATH.exists():
        raise Ov2Error(f"{_LIBPATH} is missing: run `python -m ov2slam_b200.build` "
                       "(there is no CPU fallback for the hot paths)")
    lib = C.CDLL(str(_LIBPATH))
    vp, i32, sz = C.c_void_p, C.c_int, C.c_size_t
    lib.ov2_create.argtypes = [i32, C.POINTER(vp)]
    lib.ov2_destroy.argtypes = [vp]
    lib.ov2_destroy.restype = None
    lib.ov2_last_error.argtypes = [vp]
    lib.ov2_last_error.restype = C.c_char_p
    lib.ov2_version.restype = C.c_char_p
    lib.ov2_set_stream.argtypes = [vp, vp]
    lib.ov2_sync.argtypes = [vp]
    lib.ov2_batch_begin.argtypes = [vp]
    lib.ov2_batch_end.argtypes = [vp]
    lib.ov2_host_alloc.argtypes = [vp, sz, C.POINTER(vp)]
    lib.ov2_host_free.argtypes = [vp, vp]
    lib.ov2_launch_count.argtypes = [vp]
    lib.ov2_launch_count.restype = C.c_uint64
    lib.ov2_profile_enable.argtypes = [vp, i32]
    lib.ov2_profile_query.argtypes = [vp, i32, C.c_char_p, i32, C.POINTER(C.c_double), C.POINTER(C.c_uint64)]
    lib.ov2_pyr_create.argtypes = [vp, i32, i32, i32, i32, C.POINTER(vp)]
    lib.ov2_pyr_destroy.argtypes = [vp]
    lib.ov2_pyr_destroy.restype = None
    lib.ov2_pyr_build.argtypes = [vp, vp, vp, sz, sz, i32, i32]
    lib.ov2_pyr_download.argtypes = [vp, vp, i32, i32, vp, C.POINTER(i32), C.POINTER(i32)]
    lib.ov2_clahe.argtypes = [vp, vp, vp, i32, i32, sz, sz, i32, C.c_double, i32, i32]
    lib.ov2_preprocess.argtypes = [vp, vp, vp, i32, i32, i32, C.c_double, i32, i32]
    lib.ov2_fb_klt.argtypes = [vp, vp, vp, C.POINTER(KltParams), i32, vp, i32, i32, vp, i32, vp, vp, vp]
    lib.ov2_grid_fast.argtypes = [vp, vp, i32, i32, i32, vp, vp, vp, i32, vp, vp, vp, i32]
    lib.ov2_detect_single_scale.argtypes = [vp, vp, i32, i32, i32, vp, vp, vp, vp, i32, vp, vp, vp, i32]
    lib.ov2_pnp_solve.argtypes = [vp, i32, vp, vp, vp, vp, vp, vp, i32, C.c_float, i32, i32, vp, vp, vp]
    lib.ov2_debug_fast_cells.argtypes = [vp, vp, i32, i32, i32, vp, vp, i32, C.POINTER(i32)]
    lib.ov2_describe.argtypes = [vp, vp, i32, vp, i32, i32, vp, vp, vp]
    lib.ov2_describe_config.argtypes = [vp, i32, vp]
    lib.ov2_line_min_sad.argtypes = [vp, vp, vp, i32, i32, vp, i32, i32, vp, i32, i32, vp, vp]
    lib.ov2_match_to_map.argtypes = [vp, C.POINTER(MatchProblem), vp, vp, vp, vp]
    lib.ov2_frontend_step.argtypes = [vp, vp, vp, C.POINTER(FrontendStepArgs)]
    lib.ov2_localba_solve.argtypes = [vp, C.POINTER(BaProblem), C.POINTER(BaOpts), C.POINTER(BaResult), vp]
    lib.ov2_localba_solve_sharded.argtypes = [vp, C.POINTER(BaProblem), C.POINTER(BaOpts), C.POINTER(BaResult), vp,
                                              ALLREDUCE_FN, vp, i32]
    lib.ov2_localba_solve_batch.argtypes = [vp, i32, C.POINTER(BaProblem), C.POINTER(BaOpts), C.POINTER(BaResult), vp]
    lib.ov2_localba_request_stop.argtypes = [vp, i32]
    lib.ov2_ba_comm_create.argtypes = [vp, i32, i32, C.POINTER(vp)]
    lib.ov2_ba_comm_handle.argtypes = [vp, vp, sz]
    lib.ov2_ba_comm_connect.argtypes = [vp, vp, sz]
    lib.ov2_ba_comm_connect_local.argtypes = [vp, C.POINTER(vp)]
    lib.ov2_ba_comm_destroy.argtypes = [vp]
    lib.ov2_ba_comm_destroy.restype = None
    lib.ov2_localba_solve_p2p.argtypes = [vp, vp, C.POINTER(BaProblem), C.POINTER(BaOpts), C.POINTER(BaResult), vp]
    _lib = lib
    return lib


def _ptr(a):
    """Raw address of a numpy array (host), a torch tensor (host or CUDA), an int, or None."""
    if a is None:
        return None
    if isinstance(a, int):
        return a
    if isinstance(a, np.ndarray):
        if not a.flags["C_CONTIGUOUS"]:
            raise Ov2Error("array must be C-contiguous")
        return a.ctypes.data
    if hasattr(a, "data_ptr"):
        if not a.is_contiguous():
            raise Ov2Error("tensor must be contiguous")
        return a.data_ptr()
    raise Ov2Error(f"unsupported array type {type(a)}")


class Context:
    """ov2_ctx: one CUDA device + stream + scratch arena.  Not re-entrant."""

    def __init__(self, device: int = 0, stream: int | None = None):
        self.lib = load()
        h = C.c_void_p()
        st = self.lib.ov2_create(int(device), C.byref(h))
        if st != OV2_OK:
            raise Ov2Error(f"ov2_create(device={device}) failed: {STATUS_NAMES.get(st, st)} "
                           "(the hot paths run on a CUDA device only; there is no CPU fallback)")
        self.h = h
        self.device = device
        self._pyramids = []   # weak refs: pyramids must be destroyed before the context
        if stream is not None:
            self.check(self.lib.ov2_set_stream(self.h, C.c_void_p(stream)))

    def check(self, st: int):
        if st != OV2_OK:
            msg = self.lib.ov2_last_error(self.h)
            raise Ov2Error(f"{STATUS_NAMES.get(st, st)}: {msg.decode() if msg else ''}")

    def sync(self):
        self.check(self.lib.ov2_sync(self.h))

    def batch_begin(self):
        self.check(self.lib.ov2_batch_begin(self.h))

    def batch_end(self):
        self.check(self.lib.ov2_batch_end(self.h))

    def launch_count(self) -> int:
        return int(self.lib.ov2_launch_count(self.h))

    def profile(self, on: bool):
        self.check(self.lib.ov2_profile_enable(self.h, 1 if on else 0))

    def profile_report(self) -> dict:
        """{kernel name: (total ms, launches)} accumulated since profile(True)."""
        out = {}
        buf = C.create_string_buffer(64)
        ms, n = C.c_double(), C.c_uint64()
        i = 0
        while self.lib.ov2_profile_query(self.h, i, buf, 64, C.byref(ms), C.byref(n)):
            out[buf.value.decode()] = (ms.value, int(n.value))
            i += 1
        return out

    def close(self):
        if self.h:
            for r in self._pyramids:
                p = r()
                if p is not None:
                    p.close()
            self._pyramids = []
            self.lib.ov2_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Pyramid:
    """ov2_pyr: device-resident pyramids of a batch of frames (P)."""

    def __init__(self, ctx: Context, batch: int, width: int, height: int, nlevels_extra: int = 3):
        self.ctx = ctx
        self.batch, self.w, self.h, self.nlev = batch, width, height, nlevels_extra + 1
        h = C.c_void_p()
        ctx.check(ctx.lib.ov2_pyr_create(ctx.h, batch, width, height, nlevels_extra, C.byref(h)))
        self.h_ = h
        self._keepalive = None
        ctx._pyramids.append(weakref.ref(self))

    def build(self, images, first: int = 0, count: int | None = None, row_stride=None, frame_stride=None):
        """images: (count, H, W) uint8 numpy array (host) or CUDA torch tensor (used in place)."""
        if count is None:
            count = images.shape[0] if images.ndim == 3 else 1   # (raw int addresses need an explicit count)
        rs = int(row_stride if row_stride is not None else self.w)
        fs = int(frame_stride if frame_stride is not None else rs * self.h)
        self.ctx.check(self.ctx.lib.ov2_pyr_build(self.ctx.h, self.h_, _ptr(images), rs, fs, first, count))
        if hasattr(images, "data_ptr"):
            self._keepalive = images

    def download(self, frame: int, level: int) -> np.ndarray:
        lw, lh = self.w, self.h
        for _ in range(level):
            lw, lh = (lw + 1) // 2, (lh + 1) // 2
        out = np.empty((lh, lw), np.uint8)
        a, b = C.c_int(), C.c_int()
        self.ctx.check(self.ctx.lib.ov2_pyr_download(self.ctx.h, self.h_, frame, level, out.ctypes.data,
                                                     C.byref(a), C.byref(b)))
        assert (a.value, b.value) == (lw, lh)
        return out

    def close(self):
        if self.h_ and self.ctx.h:
            self.ctx.lib.ov2_pyr_destroy(self.h_)
        self.h_ = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def frontend_step(ctx: Context, prev: "Pyramid", cur: "Pyramid", args: FrontendStepArgs):
    """ov2_frontend_step: pyramids, fb-KLT, grid FAST + subpix and both descriptor passes for a batch of
    frame pairs in one call (one sync)."""
    ctx.check(ctx.lib.ov2_frontend_step(ctx.h, prev.h_, cur.h_, C.byref(args)))


def clahe(ctx: Context, src, dst, width: int, height: int, count: int = 1, clip_limit: float = 3.0,
          tiles=None, row_stride=None, frame_stride=None):
    """cv::CLAHE::apply on `count` images (numpy or CUDA tensors); tiles default to the reference's
    Size(W/50, H/50) (ov2slam.cpp:85-89)."""
    tx, ty = tiles if tiles is not None else (width // 50, height // 50)
    rs = int(row_stride if row_stride is not None else width)
    fs = int(frame_stride if frame_stride is not None else rs * height)
    ctx.check(ctx.lib.ov2_clahe(ctx.h, _ptr(src), _ptr(dst), width, height, rs, fs, count, float(clip_limit), tx, ty))


def preprocess(ctx: Context, raw: "Pyramid", out: "Pyramid", first: int = 0, count: int | None = None, use_clahe: bool = True,
               clip_limit: float = 3.0, tiles=None):
    """VisualFrontEnd::preprocessImage (visual_front_end.cpp:1143-1177): CLAHE of the raw level 0 into `out`
    (tiles default to the reference's Size(W/50, H/50)) + the pyramid levels of `out`."""
    tx, ty = tiles if tiles is not None else (raw.w // 50, raw.h // 50)
    ctx.check(ctx.lib.ov2_preprocess(ctx.h, raw.h_, out.h_, int(first), int(raw.batch if count is None else count),
                                     1 if use_clahe else 0, float(clip_limit), int(tx), int(ty)))


class FeatureTracker:
    """Mirror of the reference's FeatureTracker (include/feature_tracker.hpp:33-56)."""

    def __init__(self, ctx: Context, nmax_iter: int = 30, fmax_px_precision: float = 0.01):
        self.ctx = ctx
        self.nmax_iter = nmax_iter
        self.fmax_px_precision = float(np.float32(fmax_px_precision))

    def fb_klt_tracking(self, prev: Pyramid, cur: Pyramid, nwinsize, nbpyrlvl, ferr, fmax_fbklt_dist,
                        kps, priors_inout, status_out, n=None, frame_idx=None, first_frame=0, per_frame=None):
        """fbKltTracking over a (ragged or fixed-stride) batch.  nbpyrlvl: int or per-keypoint uint8
        array.  kps / priors_inout: (n, 2) float32; status_out: (n,) uint8.  Arrays may be numpy
        (host) or CUDA tensors (device)."""
        if n is None:
            n = int(kps.shape[0])
        prm = KltParams(int(nwinsize), int(self.nmax_iter), self.fmax_px_precision, float(ferr), float(fmax_fbklt_dist))
        if isinstance(nbpyrlvl, (int, np.integer)) and int(nbpyrlvl) < 64:
            lv_ptr, lv_all = None, int(nbpyrlvl)       # a pyramid depth; larger ints are raw addresses
        else:
            lv_ptr, lv_all = _ptr(nbpyrlvl), 0
        if frame_idx is None and per_frame is None:
            per_frame = max(n, 1)
        self.ctx.check(self.ctx.lib.ov2_fb_klt(self.ctx.h, prev.h_, cur.h_, C.byref(prm), n, _ptr(frame_idx),
                                               int(first_frame), int(per_frame or 0), lv_ptr, lv_all,
                                               _ptr(kps), _ptr(priors_inout), _ptr(status_out)))

    def line_min_sad(self, left: Pyramid, right: Pyramid, level: int, pts, nwinsize, goleft, xprior_out, l1err_out,
                     n=None, frame_idx=None, first_frame=0, per_frame=None):
        """getLineMinSAD (feature_tracker.cpp:138-204) for a batch of points of pyramid level `level` (the stereo prior
        MapManager::stereoMatching computes per keypoint, map_manager.cpp:417-431): xprior_out / l1err_out (n,) float32."""
        if n is None:
            n = int(pts.shape[0])
        if frame_idx is None and per_frame is None:
            per_frame = max(n, 1)
        self.ctx.check(self.ctx.lib.ov2_line_min_sad(self.ctx.h, left.h_, right.h_, int(level), n, _ptr(frame_idx), int(first_frame),
                                                     int(per_frame or 0), _ptr(pts), int(nwinsize), 1 if goleft else 0,
                                                     _ptr(xprior_out), _ptr(l1err_out)))


class FeatureExtractor:
    """Mirror of the reference's FeatureExtractor (include/feature_extractor.hpp:31-55) for the
    hot-path methods detectGridFAST and describeBRIEF."""

    def __init__(self, ctx: Context, nmaxpts: int = 0, nmaxdist: int = 50, dmaxquality: float = 0.0, nfast_th: int = 10):
        self.ctx = ctx
        self.nmaxpts_, self.nmaxdist_, self.dmaxquality_, self.nfast_th_ = nmaxpts, nmaxdist, dmaxquality, nfast_th

    def detect_grid_fast(self, pyr: Pyramid, ncellsize: int, first: int, count: int, fast_th_inout,
                         out_pts, out_counts, curkp_offsets=None, curkps=None, out_pts_int=None,
                         max_per_frame=None, do_subpix=True):
        if max_per_frame is None:
            max_per_frame = (pyr.h // ncellsize) * (pyr.w // ncellsize)
        self.ctx.check(self.ctx.lib.ov2_grid_fast(self.ctx.h, pyr.h_, first, count, ncellsize,
                                                  _ptr(curkp_offsets), _ptr(curkps), _ptr(fast_th_inout),
                                                  int(max_per_frame), _ptr(out_pts), _ptr(out_counts),
                                                  _ptr(out_pts_int), 1 if do_subpix else 0))

    def detect_single_scale(self, pyr: Pyramid, ncellsize: int, first: int, count: int, quality_inout,
                            out_pts, out_counts, curkp_offsets=None, curkps=None, roi=None, out_pts_int=None,
                            max_per_frame=None, do_subpix=True):
        """detectSingleScale (feature_extractor.cpp:288-440) for frames [first, first+count); quality_inout is
        the float64 dmaxquality_ state per frame stream; roi = (x, y, w, h) or None (whole image)."""
        if max_per_frame is None:
            max_per_frame = (pyr.h // ncellsize) * (pyr.w // ncellsize)
        roi_arr = None if roi is None else np.ascontiguousarray(roi, np.int32)
        self.ctx.check(self.ctx.lib.ov2_detect_single_scale(self.ctx.h, pyr.h_, first, count, ncellsize,
                                                            _ptr(curkp_offsets), _ptr(curkps), _ptr(roi_arr),
                                                            _ptr(quality_inout), int(max_per_frame), _ptr(out_pts),
                                                            _ptr(out_counts), _ptr(out_pts_int), 1 if do_subpix else 0))

    def detect_single_scale_frame(self, pyr: Pyramid, frame: int, ncellsize: int, vcurkps, roi=None):
        """Single-frame convenience with the reference's signature shape; carries dmaxquality_ like the class."""
        ncell = (pyr.h // ncellsize) * (pyr.w // ncellsize)
        cur = np.ascontiguousarray(vcurkps, np.float32).reshape(-1, 2)
        off = np.array([0, len(cur)], np.int32)
        q = np.array([self.dmaxquality_], np.float64)
        pts = np.empty((ncell, 2), np.float32)
        ipts = np.empty((ncell, 2), np.int32)
        cnt = np.zeros(1, np.int32)
        self.detect_single_scale(pyr, ncellsize, frame, 1, q, pts, cnt, off, cur if len(cur) else None, roi, ipts)
        self.dmaxquality_ = float(q[0])
        return pts[:cnt[0]].copy(), ipts[:cnt[0]].copy()

    def detect_grid_fast_frame(self, pyr: Pyramid, frame: int, ncellsize: int, vcurkps):
        """Single-frame convenience with the reference's signature shape:
        detectGridFAST(im, ncellsize, vcurkps, roi) -> points; carries nfast_th_ like the class does."""
        ncell = (pyr.h // ncellsize) * (pyr.w // ncellsize)
        cur = np.ascontiguousarray(vcurkps, np.float32).reshape(-1, 2)
        off = np.array([0, len(cur)], np.int32)
        th = np.array([self.nfast_th_], np.int32)
        pts = np.empty((ncell, 2), np.float32)
        ipts = np.empty((ncell, 2), np.int32)
        cnt = np.zeros(1, np.int32)
        self.detect_grid_fast(pyr, ncellsize, frame, 1, th, pts, cnt, off, cur if len(cur) else None, ipts)
        self.nfast_th_ = int(th[0])
        return pts[:cnt[0]].copy(), ipts[:cnt[0]].copy()

    def debug_fast_cells(self, pyr: Pyramid, frame: int, ncellsize: int, fast_th: int):
        """Stage F1 only: list per cell of (x, y, response) candidates (cell-local, scan order)."""
        ncell = (pyr.h // ncellsize) * (pyr.w // ncellsize)
        cand = np.zeros((ncell, 128), np.uint32)
        cn = np.zeros(ncell, np.int32)
        cap = C.c_int()
        self.ctx.check(self.ctx.lib.ov2_debug_fast_cells(self.ctx.h, pyr.h_, frame, ncellsize, int(fast_th),
                                                         cand.ctypes.data, cn.ctypes.data, 128, C.byref(cap)))
        flat = cand.reshape(-1)[:ncell * cap.value].reshape(ncell, cap.value)
        return [[(int(v & 255), int((v >> 8) & 255), float(v >> 16)) for v in flat[c, :cn[c]]] for c in range(ncell)]

    DESC_ORB_FALLBACK, DESC_BRIEF32 = 0, 1

    def describe_config(self, mode: int, pairs=None):
        """ov2_describe_config: DESC_ORB_FALLBACK (reference built without opencv_contrib, the default here) or
        DESC_BRIEF32 with the int8[256][4] = (y0, x0, y1, x1) test pairs of opencv_contrib's generated_32.i."""
        keep = None if pairs is None else np.ascontiguousarray(pairs, np.int8).reshape(256, 4)
        self.ctx.check(self.ctx.lib.ov2_describe_config(self.ctx.h, int(mode), None if keep is None else keep.ctypes.data))

    def describe_brief(self, pyr: Pyramid, pts, desc_out, valid_out, n=None, frame_idx=None, first_frame=0,
                       per_frame=None):
        if n is None:
            n = int(pts.shape[0])
        if frame_idx is None and per_frame is None:
            per_frame = max(n, 1)
        self.ctx.check(self.ctx.lib.ov2_describe(self.ctx.h, pyr.h_, n, _ptr(frame_idx), int(first_frame),
                                                 int(per_frame or 0), _ptr(pts), _ptr(desc_out), _ptr(valid_out)))


def _stereo_ptrs(pb: dict, keep: dict):
    """(obs_type, Kr, Trl) pointers for a stereo window, (None, None, None) for a mono one."""
    if pb.get("obs_type") is None:
        return None, None, None
    keep["obs_type"] = np.ascontiguousarray(pb["obs_type"], np.uint8)
    keep["Kr"] = np.ascontiguousarray(pb["Kr"], np.float64)
    keep["Trl"] = np.ascontiguousarray(pb["Trl"], np.float64)
    return keep["obs_type"].ctypes.data, keep["Kr"].ctypes.data, keep["Trl"].ctypes.data


# Capacity of one Optimizer.local_ba / ov2_localba_solve window (include/ov2b200.h): optimised and total keyframes.  Windows
# of up to 64 optimised keyframes run the small-window kernel, larger ones the large-window kernel; batches and the
# multi-GPU solves keep 64 / 256.
OV2_BA_MAX_OPT_KEYFRAMES = 1024
OV2_BA_MAX_KEYFRAMES = 4096
OV2_BA_SMALL_MAX_OPT_KEYFRAMES = 64
OV2_BA_SMALL_MAX_KEYFRAMES = 256

DEFAULT_BA_OPTS = dict(max_iters_robust=5, max_iters_refine=10, huber_th=5.9915, function_tolerance=1e-3,
                       use_robust=1, apply_l2_after_robust=1, refine_loss=-1)


class MultiViewGeometry:
    """Mirror of the reference's static MultiViewGeometry::ceresPnP (multi_view_geometry.cpp:492-588), batched."""

    def __init__(self, ctx: "Context"):
        self.ctx = ctx

    def ceres_pnp_batch(self, offsets, unpx, wpts, K, poses_inout, nmaxiter=5, chi2th=5.9915, use_robust=True,
                        apply_l2_after_robust=True, scales=None):
        """offsets int32[nprob+1] (host), unpx float64[N,2], wpts float64[N,3], K float64[nprob,4],
        poses_inout float64[nprob,7] (Twc = t, q xyzw).  Returns (success uint8[nprob], outlier flags uint8[N],
        LM iterations int32[nprob])."""
        offsets = np.ascontiguousarray(offsets, np.int32)
        nprob = len(offsets) - 1
        n = int(offsets[-1])
        flags = np.zeros(max(n, 1), np.uint8)
        success = np.zeros(max(nprob, 1), np.uint8)
        its = np.zeros(max(nprob, 1), np.int32)
        self.ctx.check(self.ctx.lib.ov2_pnp_solve(self.ctx.h, nprob, offsets.ctypes.data, _ptr(unpx), _ptr(wpts), _ptr(scales),
                                                  _ptr(K), _ptr(poses_inout), int(nmaxiter), float(chi2th),
                                                  1 if use_robust else 0, 1 if apply_l2_after_robust else 0,
                                                  flags.ctypes.data, success.ctypes.data, its.ctypes.data))
        return success[:nprob], flags[:n], its[:nprob]

    def ceres_pnp(self, vunkps, vwpts, Twc, nmaxiter, chi2th, buse_robust, bapply_l2_after_robust, fx, fy, cx, cy, vscales=None):
        """Single problem with the reference's argument order.  Returns (success, Twc_out, voutliersidx)."""
        unpx = np.ascontiguousarray(vunkps, np.float64).reshape(-1, 2)
        wpts = np.ascontiguousarray(vwpts, np.float64).reshape(-1, 3)
        pose = np.ascontiguousarray(Twc, np.float64).reshape(1, 7).copy()
        K = np.array([[fx, fy, cx, cy]], np.float64)
        sc = None if vscales is None else np.ascontiguousarray(vscales, np.int32)
        ok, flags, _ = self.ceres_pnp_batch(np.array([0, len(unpx)], np.int32), unpx, wpts, K, pose, nmaxiter, chi2th,
                                            buse_robust, bapply_l2_after_robust, sc)
        return bool(ok[0]), pose[0], np.nonzero(flags)[0]


class Optimizer:
    """Mirror of the solve part of the reference's Optimizer::localBA (optimizer.cpp:436-735)."""

    def __init__(self, ctx: Context):
        self.ctx = ctx

    def local_ba(self, pb: dict, **opts):
        """pb: dict of flat arrays as produced by synth.make_ba_problem (poses / inverse depths are
        updated in place).  Returns (result dict, outlier flags uint8[nobs])."""
        o = dict(DEFAULT_BA_OPTS)
        o.update(opts)
        bo = BaOpts(**o)
        keep = {}
        p = _ba_problem_struct(pb, keep)
        nobs = len(keep["obs_cam"])
        res = BaResult()
        flags = np.zeros(nobs, np.uint8)
        self.ctx.check(self.ctx.lib.ov2_localba_solve(self.ctx.h, C.byref(p), C.byref(bo), C.byref(res), flags.ctypes.data))
        if keep["pose"] is not pb["pose"]:
            pb["pose"][...] = keep["pose"]
        if keep["lm_invdepth"] is not pb["lm_invdepth"]:
            pb["lm_invdepth"][...] = keep["lm_invdepth"]
        return {f: getattr(res, f) for f, _ in BaResult._fields_}, flags


_BA_KEYS = ("K", "pose", "pose_const", "lm_anchor_cam", "lm_anchor_px", "lm_invdepth", "obs_cam", "obs_lm", "obs_px")
_BA_RES_DTYPE = np.dtype([("iters_robust", np.int32), ("iters_refine", np.int32), ("initial_cost", np.float64), ("final_cost", np.float64),
                          ("n_outliers_first", np.int32), ("n_outliers_second", np.int32), ("termination", np.int32), ("_pad", np.int32)])
assert _BA_RES_DTYPE.itemsize == C.sizeof(BaResult)


def _c_array(a):
    """a itself when it already is a C-contiguous ndarray (the usual case: no copy, no new object), a contiguous copy otherwise."""
    return a if isinstance(a, np.ndarray) and a.flags.c_contiguous else np.ascontiguousarray(a)


def _addr(a: np.ndarray) -> int:
    """Address of a contiguous ndarray's first byte (3x cheaper than a.ctypes.data; read-only or empty arrays take that route)."""
    try:
        return C.addressof(C.c_char.from_buffer(a))
    except (TypeError, ValueError):
        return a.ctypes.data


def _ba_problem_struct(pb: dict, keep: dict) -> BaProblem:
    for k in _BA_KEYS:
        keep[k] = _c_array(pb[k])
    assert keep["pose"].dtype == np.float64 and keep["obs_px"].dtype == np.float64 and keep["lm_invdepth"].dtype == np.float64
    assert keep["obs_cam"].dtype == np.int32 and keep["obs_lm"].dtype == np.int32 and keep["pose_const"].dtype == np.uint8
    return BaProblem(len(keep["pose"]), len(keep["lm_invdepth"]), len(keep["obs_cam"]),
                     *[_addr(keep[k]) for k in _BA_KEYS], *_stereo_ptrs(pb, keep))


def local_ba_batch(ctx: Context, pbs: list, **opts):
    """ov2_localba_solve_batch: K windows (dicts as Optimizer.local_ba takes) in one launch; poses / inverse depths are
    updated in place.  Returns (list of result dicts, list of flag arrays)."""
    o = dict(DEFAULT_BA_OPTS)
    o.update(opts)
    bo = BaOpts(**o)
    n = len(pbs)
    keeps = [dict() for _ in pbs]
    arr = (BaProblem * n)(*[_ba_problem_struct(pb, kp) for pb, kp in zip(pbs, keeps)])
    res = (BaResult * n)()
    nobs = [len(kp["obs_cam"]) for kp in keeps]
    offs = np.concatenate([[0], np.cumsum([max(v, 1) for v in nobs])]).astype(np.int64)
    allflags = np.zeros(int(offs[-1]), np.uint8)                      # one buffer, one slice per window
    base = _addr(allflags)
    fl = (C.c_void_p * n)(*[base + int(v) for v in offs[:-1]])
    ctx.check(ctx.lib.ov2_localba_solve_batch(ctx.h, n, arr, C.byref(bo), res, fl))
    for pb, kp in zip(pbs, keeps):
        if kp["pose"] is not pb["pose"]:
            pb["pose"][...] = kp["pose"]
        if kp["lm_invdepth"] is not pb["lm_invdepth"]:
            pb["lm_invdepth"][...] = kp["lm_invdepth"]
    rec = np.frombuffer(res, dtype=_BA_RES_DTYPE, count=n)
    names = [f for f, _ in BaResult._fields_]
    cols = [rec[f].tolist() for f in names]
    return ([dict(zip(names, row)) for row in zip(*cols)],
            [allflags[int(offs[i]):int(offs[i]) + nobs[i]] for i in range(n)])


def match_to_map(ctx: Context, sc: dict):
    """Mapper::matchToMap (mapper.cpp:576-774) on a flattened scene (dict as ov2slam_b200.synth.make_match_scene builds it):
    returns (best_kp int32[ncand], best_dist float32[ncand], kp_match int32[nkps], kp_dist float32[nkps])."""
    keep = {}

    def arr(k, dt):
        keep[k] = np.ascontiguousarray(sc[k], dt)
        return keep[k].ctypes.data if keep[k].size else None

    p = MatchProblem()
    p.Tcw[:] = [float(v) for v in np.asarray(sc["Tcw"], np.float64).reshape(-1)]
    p.K[:] = [float(v) for v in sc["K"]]
    p.dist = arr("dist", np.float64) if sc.get("dist") is not None else None
    p.img_w, p.img_h, p.ncellsize, p.nbwcells = int(sc["img_w"]), int(sc["img_h"]), int(sc["ncellsize"]), int(sc["nbwcells"])
    p.ncells = len(sc["cell_ptr"]) - 1
    p.cell_ptr, p.cell_kp = arr("cell_ptr", np.int32), arr("cell_kp", np.int32)
    p.nkps = len(sc["kp_px"])
    p.kp_px, p.kp_lm = arr("kp_px", np.float32), arr("kp_lm", np.int32)
    p.nmps = len(sc["mp_xyz"])
    p.mp_xyz, p.mp_desc_ptr = arr("mp_xyz", np.float64), arr("mp_desc_ptr", np.int32)
    p.ndesc = len(sc["desc"])
    p.desc, p.mp_kfmask = arr("desc", np.uint8), arr("mp_kfmask", np.uint64)
    p.mp_obs_ptr = arr("mp_obs_ptr", np.int32)
    p.nobs = len(sc["obs_kf"])
    p.obs_kf, p.obs_px = arr("obs_kf", np.int32), arr("obs_px", np.float32)
    p.nkfs = len(np.asarray(sc["kf_Tcw"]).reshape(-1, 12))
    p.kf_Tcw = arr("kf_Tcw", np.float64)
    p.ncand = len(sc["cand_mp"])
    p.cand_mp = arr("cand_mp", np.int32)
    p.dmaxpxdist, p.fdistratio, p.view_th = float(sc["dmaxpxdist"]), float(sc["fdistratio"]), float(sc["view_th"])
    best_kp = np.full(max(p.ncand, 1), -1, np.int32)
    best_dist = np.zeros(max(p.ncand, 1), np.float32)
    kp_match = np.full(max(p.nkps, 1), -1, np.int32)
    kp_dist = np.zeros(max(p.nkps, 1), np.float32)
    ctx.check(ctx.lib.ov2_match_to_map(ctx.h, C.byref(p), best_kp.ctypes.data, best_dist.ctypes.data, kp_match.ctypes.data, kp_dist.ctypes.data))
    return best_kp[:p.ncand], best_dist[:p.ncand], kp_match[:p.nkps], kp_dist[:p.nkps]


def request_stop_local_ba(ctx: Context, stop: bool = True):
    """Optimizer::signalStopLocalBA (optimizer.cpp:2334-2343): ask the solve on `ctx` to skip the refinement."""
    ctx.check(ctx.lib.ov2_localba_request_stop(ctx.h, 1 if stop else 0))


# ----------------------------------------------------------------------------- multi-GPU local BA
class BaComm:
    """ov2_ba_comm: this rank's exchange buffer + the peers' buffers (CUDA IPC between processes, direct pointers inside
    one process).  connect_torch() exchanges the IPC handles with torch.distributed (any backend)."""

    HANDLE = 64

    def __init__(self, ctx: Context, rank: int, world: int):
        self.ctx, self.rank, self.world = ctx, rank, world
        h = C.c_void_p()
        ctx.check(ctx.lib.ov2_ba_comm_create(ctx.h, rank, world, C.byref(h)))
        self.h = h

    def handle(self) -> bytes:
        buf = C.create_string_buffer(self.HANDLE)
        self.ctx.check(self.ctx.lib.ov2_ba_comm_handle(self.h, buf, self.HANDLE))
        return buf.raw

    def connect(self, handles: list):
        assert len(handles) == self.world and all(len(x) == self.HANDLE for x in handles)
        blob = b"".join(handles)
        self.ctx.check(self.ctx.lib.ov2_ba_comm_connect(self.h, blob, self.HANDLE))

    def connect_torch(self, dist, torch, group=None):
        if self.world == 1:
            return
        mine = torch.frombuffer(bytearray(self.handle()), dtype=torch.uint8).clone()
        dev = "cuda" if dist.get_backend(group) == "nccl" else "cpu"
        mine = mine.to(dev)
        got = [torch.empty_like(mine) for _ in range(self.world)]
        dist.all_gather(got, mine, group=group)
        self.connect([bytes(g.cpu().numpy().tobytes()) for g in got])

    @staticmethod
    def connect_local(comms: list):
        arr = (C.c_void_p * len(comms))(*[c.h for c in comms])
        for c in comms:
            c.ctx.check(c.ctx.lib.ov2_ba_comm_connect_local(c.h, arr))

    def local_ba(self, shard: dict, **opts):
        """ov2_localba_solve_p2p on this rank's shard (collective)."""
        o = dict(DEFAULT_BA_OPTS)
        o.update(opts)
        bo = BaOpts(**o)
        keep = {}
        p = _ba_problem_struct(shard, keep)
        res = BaResult()
        flags = np.zeros(max(len(keep["obs_cam"]), 1), np.uint8)
        self.ctx.check(self.ctx.lib.ov2_localba_solve_p2p(self.ctx.h, self.h, C.byref(p), C.byref(bo), C.byref(res), flags.ctypes.data))
        shard["pose"][...] = keep["pose"]
        shard["lm_invdepth"][...] = keep["lm_invdepth"]
        return {f: getattr(res, f) for f, _ in BaResult._fields_}, flags[:len(keep["obs_cam"])]

    def close(self):
        if self.h and self.ctx.h:
            self.ctx.lib.ov2_ba_comm_destroy(self.h)
        self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def partition_ba_problem(pb: dict, world: int):
    """Split a flat localBA window into `world` shards by LANDMARK (all observations of a landmark
    stay on one rank, so the per-landmark Schur elimination is local; SURVEY.md 8e), balancing the
    number of observations greedily.  Every shard keeps all cameras.  Returns a list of
    (shard dict, landmark index array, observation index array)."""
    npts, nobs = len(pb["lm_invdepth"]), len(pb["obs_cam"])
    counts = np.bincount(pb["obs_lm"], minlength=npts)
    order = np.argsort(-counts, kind="stable")
    load = np.zeros(world, np.int64)
    owner = np.empty(npts, np.int64)
    for l in order:                      # longest-processing-time greedy
        r = int(np.argmin(load))
        owner[l] = r
        load[r] += counts[l] + 1
    shards = []
    for r in range(world):
        lms = np.nonzero(owner == r)[0]                      # ascending -> observations stay sorted
        remap = -np.ones(npts, np.int64)
        remap[lms] = np.arange(len(lms))
        obs = np.nonzero(owner[pb["obs_lm"]] == r)[0]
        sh = dict(K=pb["K"].copy(), pose=pb["pose"].copy(), pose_const=pb["pose_const"].copy(),
                  lm_anchor_cam=np.ascontiguousarray(pb["lm_anchor_cam"][lms]),
                  lm_anchor_px=np.ascontiguousarray(pb["lm_anchor_px"][lms]),
                  lm_invdepth=np.ascontiguousarray(pb["lm_invdepth"][lms]),
                  obs_cam=np.ascontiguousarray(pb["obs_cam"][obs]),
                  obs_lm=np.ascontiguousarray(remap[pb["obs_lm"][obs]].astype(np.int32)),
                  obs_px=np.ascontiguousarray(pb["obs_px"][obs]))
        if pb.get("obs_type") is not None:
            sh.update(obs_type=np.ascontiguousarray(pb["obs_type"][obs]), Kr=pb["Kr"].copy(), Trl=pb["Trl"].copy())
        shards.append((sh, lms, obs))
    return shards


class _CudaView:
    """Zero-copy view of raw device memory for torch.as_tensor (CUDA array interface v2)."""

    def __init__(self, ptr: int, count: int):
        self.__cuda_array_interface__ = {"shape": (count,), "typestr": "<f8", "data": (ptr, False), "version": 2}


def make_torch_allreduce(dist, torch, group=None):
    """ov2_allreduce_fn that sums the buffer over the process group with torch.distributed
    (NCCL over NVLink for device buffers; gloo for the CPU tests, where `buf` is host memory)."""
    def _fn(user, buf, count, stream):
        try:
            if torch.cuda.is_available() and dist.get_backend(group) == "nccl":
                t = torch.as_tensor(_CudaView(buf, count), device="cuda")
                s = torch.cuda.ExternalStream(stream) if stream else torch.cuda.current_stream()
                with torch.cuda.stream(s):
                    dist.all_reduce(t, group=group)
            else:
                a = np.ctypeslib.as_array(C.cast(buf, C.POINTER(C.c_double)), shape=(count,))
                t = torch.from_numpy(a)
                dist.all_reduce(t, group=group)
            return 0
        except Exception as e:  # never let an exception cross the C boundary
            print("[ov2b200] allreduce callback failed:", e, flush=True)
            return 1
    return ALLREDUCE_FN(_fn)


def local_ba_sharded(ctx: Context, shard: dict, allreduce_cb, rank: int, **opts):
    """ov2_localba_solve_sharded on this rank's shard; poses come back identical on every rank,
    inverse depths / flags are the shard's own."""
    o = dict(DEFAULT_BA_OPTS)
    o.update(opts)
    bo = BaOpts(**o)
    keep = {k: np.ascontiguousarray(shard[k]) for k in
            ("K", "pose", "pose_const", "lm_anchor_cam", "lm_anchor_px", "lm_invdepth", "obs_cam", "obs_lm", "obs_px")}
    p = BaProblem(len(keep["pose"]), len(keep["lm_invdepth"]), len(keep["obs_cam"]),
                  *[keep[k].ctypes.data for k in ("K", "pose", "pose_const", "lm_anchor_cam", "lm_anchor_px", "lm_invdepth",
                                                  "obs_cam", "obs_lm", "obs_px")], *_stereo_ptrs(shard, keep))
    res = BaResult()
    flags = np.zeros(max(len(keep["obs_cam"]), 1), np.uint8)
    ctx.check(ctx.lib.ov2_localba_solve_sharded(ctx.h, C.byref(p), C.byref(bo), C.byref(res), flags.ctypes.data,
                                                allreduce_cb, None, int(rank)))
    shard["pose"][...] = keep["pose"]
    shard["lm_invdepth"][...] = keep["lm_invdepth"]
    return {f: getattr(res, f) for f, _ in BaResult._fields_}, flags[:len(keep["obs_cam"])]


class ShardedOptimizer:
    """Multi-GPU Optimizer::localBA (BASELINE.json configs[4]): this rank's landmark shard, poses replicated.
    mode "p2p" (default): the per-iteration sum of the reduced camera system happens inside the solve kernel over peer
    memory (ov2_localba_solve_p2p); mode "callback": round-1 path, ncclAllReduce through torch.distributed per iteration."""

    def __init__(self, ctx: Context, dist, torch, rank: int, world: int, group=None, mode: str = "p2p"):
        self.ctx, self.rank, self.world, self.mode = ctx, rank, world, mode
        if mode == "p2p":
            self.comm = BaComm(ctx, rank, world)
            self.comm.connect_torch(dist, torch, group)
        else:
            self._cb = make_torch_allreduce(dist, torch, group)

    def local_ba(self, shard: dict, **opts):
        if self.mode == "p2p":
            return self.comm.local_ba(shard, **opts)
        return local_ba_sharded(self.ctx, shard, self._cb, self.rank, **opts)

    def describe(self) -> str:
        return ("in-kernel sum of the partial reduced systems over NVLink peer memory (CUDA IPC), one persistent kernel per solve"
                if self.mode == "p2p" else "ncclAllReduce through the ov2_allreduce_fn callback (torch.distributed), host LM controller")
