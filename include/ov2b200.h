/* ov2b200.h - C ABI of the B200-native OV2SLAM hot paths (libov2b200.so).
 *
 * This is the drop-in boundary (SURVEY.md section 8b).  The reference has no FFI of its own: its
 * callers (visual_front_end.cpp, map_manager.cpp, estimator.cpp) call three C++ classes
 * directly.  The C++ shim classes in ov2slam_b200/host/ keep those class declarations
 * unchanged and forward to the entry points below; every entry point names the reference
 * interface it replaces.
 *
 * Conventions
 *   - Plain C types only.  All functions return an ov2_status (0 = OK); none throws or exits.
 *   - There is no CPU fallback: without a CUDA device ov2_create() fails with
 *     OV2_ERR_NO_DEVICE and every other call needs a context.
 *   - Array arguments may point to HOST memory (pageable or pinned) or to DEVICE memory of the
 *     context's device; the library detects which (cudaPointerGetAttributes).  Host inputs are
 *     copied H2D on the context's stream, host outputs are copied D2H and the call returns after
 *     they have landed.  With device pointers only, a call just enqueues work on the stream
 *     (use ov2_sync()).
 *   - A context is not re-entrant; use one per host thread (the reference calls
 *     fbKltTracking concurrently from the front-end and mapper threads, map_manager.cpp:510).
 *   - Batches are either "fixed stride" (frame_idx == NULL: element i belongs to frame slot
 *     first_frame + i / per_frame) or "ragged" (frame_idx[i] gives the frame slot).
 */
#ifndef OV2B200_H
#define OV2B200_H

#include <stddef.h>
#include <stdint.h>

#if defined(__GNUC__)
#define OV2_API __attribute__((visibility("default")))
#else
#define OV2_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
    OV2_OK = 0,
    OV2_ERR_NO_DEVICE = 1,   /* no CUDA device / driver: there is no CPU path */
    OV2_ERR_CUDA = 2,        /* a CUDA call failed; see ov2_last_error() */
    OV2_ERR_INVALID = 3,     /* bad argument */
    OV2_ERR_CAPACITY = 4,    /* a fixed-capacity device buffer overflowed (reported, never silent) */
    OV2_ERR_NOMEM = 5,
    OV2_ERR_NUMERIC = 6      /* BA: non-finite cost / failed factorisation */
} ov2_status;

typedef struct ov2_ctx ov2_ctx;   /* device + stream + scratch arenas */
typedef struct ov2_pyr ov2_pyr;   /* device-resident image pyramids for a batch of frames */

/* ------------------------------------------------------------------ context */
OV2_API ov2_status ov2_create(int device, ov2_ctx** out);
OV2_API void       ov2_destroy(ov2_ctx* ctx);
OV2_API const char* ov2_last_error(const ov2_ctx* ctx);      /* valid until the next call on ctx */
OV2_API const char* ov2_version(void);
/* Run the context's work on an existing stream (e.g. torch's current stream). NULL = own stream. */
OV2_API ov2_status ov2_set_stream(ov2_ctx* ctx, void* cuda_stream);
OV2_API ov2_status ov2_sync(ov2_ctx* ctx);
/* Batch mode: between ov2_batch_begin and ov2_batch_end every call on the context only ENQUEUES
 * (H2D of host inputs, kernels); host outputs are copied back and the stream is synchronised once,
 * in ov2_batch_end.  A host buffer written by one call of the batch and read by a later one (e.g.
 * the tracked positions fbKltTracking returns and describeBRIEF consumes) is served from its device
 * staging copy, so operator chains keep host-pointer semantics without round trips.  Host outputs
 * must not be read before ov2_batch_end.  (ov2_grid_fast's capacity check is skipped in a batch.) */
OV2_API ov2_status ov2_batch_begin(ov2_ctx* ctx);
OV2_API ov2_status ov2_batch_end(ov2_ctx* ctx);
/* Pinned host memory helpers (for callers that want true async H2D/D2H). */
OV2_API ov2_status ov2_host_alloc(ov2_ctx* ctx, size_t bytes, void** out);
OV2_API ov2_status ov2_host_free(ov2_ctx* ctx, void* p);
/* Number of kernels this context has launched since creation (bench.py's gpu_launches). */
OV2_API uint64_t   ov2_launch_count(const ov2_ctx* ctx);

/* Per-kernel timing with CUDA events on the launching stream (serialises launches; for
 * bench.py's roofline pass, never on during the timed benchmark region).
 * ov2_profile_query: idx-th kernel class -> name, accumulated ms, launch count; returns 0 past the end. */
OV2_API ov2_status ov2_profile_enable(ov2_ctx* ctx, int on);
OV2_API int        ov2_profile_query(const ov2_ctx* ctx, int idx, char* name_out, int name_cap, double* total_ms,
                             uint64_t* launches);

/* ------------------------------------------------------------------ P: pyramid
 * Replaces cv::buildOpticalFlowPyramid(img, pyr, Size(9,9), 3) as called by
 * VisualFrontEnd::preprocessImage (/root/reference/src/visual_front_end.cpp:1172, also :53 and
 * src/mapper.cpp:81).  The Scharr derivative planes are not materialised; the tracker
 * recomputes them on the fly from the 8-bit levels (identical values). */
OV2_API ov2_status ov2_pyr_create(ov2_ctx* ctx, int batch, int width, int height, int nlevels_extra, ov2_pyr** out);
OV2_API void       ov2_pyr_destroy(ov2_pyr* pyr);
/* Load `count` 8-bit images into frame slots [first, first+count) and build their levels.
 * `images` = host or device pointer; row r of image k starts at images + k*frame_stride + r*row_stride.
 * Device images are used in place as level 0 (they must stay alive and unchanged while the
 * pyramid is used); host images are copied into the pyramid's own level-0 storage. */
OV2_API ov2_status ov2_pyr_build(ov2_ctx* ctx, ov2_pyr* pyr, const uint8_t* images, size_t row_stride,
                         size_t frame_stride, int first, int count);
/* Copy one level of one frame slot back to host (tests). `out` holds level_w*level_h bytes, packed. */
OV2_API ov2_status ov2_pyr_download(ov2_ctx* ctx, const ov2_pyr* pyr, int frame, int level, uint8_t* out,
                            int* level_w, int* level_h);

/* ------------------------------------------------------------------ C: CLAHE
 * Replaces pclahe_->apply(img, img) with cv::createCLAHE(fclahe_val, Size(W/50, H/50))
 * (/root/reference/src/ov2slam.cpp:85-89; src/visual_front_end.cpp:1158-1160; src/mapper.cpp:75-76;
 * `use_clahe: 1`, the accurate/ configurations).  `count` 8-bit images, host or device; dst may
 * alias src only for host buffers (the device path reads src while writing dst). */
OV2_API ov2_status ov2_clahe(ov2_ctx* ctx, const uint8_t* src, uint8_t* dst, int width, int height, size_t row_stride,
                     size_t frame_stride, int count, double clip_limit, int tiles_x, int tiles_y);

/* preprocessImage as one call: VisualFrontEnd::preprocessImage (/root/reference/src/visual_front_end.cpp:1143-1177:
 * optional pclahe_->apply, prev/cur swap, cv::buildOpticalFlowPyramid) and the right-image path of Mapper::run
 * (src/mapper.cpp:75-81).  `raw` holds the untouched images (loaded with ov2_pyr_build; describeBRIEF reads the
 * raw image, src/map_manager.cpp:301-303,326-329); frames [first, first+count) of `out` receive the equalised level 0
 * (own storage) and levels 1.. built from it.  use_clahe = 0 (fast/ and average/ configurations): `out` aliases the raw
 * level 0.  The image is uploaded once however many operators read it. */
OV2_API ov2_status ov2_preprocess(ov2_ctx* ctx, const ov2_pyr* raw, ov2_pyr* out, int first, int count, int use_clahe,
                          double clip_limit, int tiles_x, int tiles_y);

/* ------------------------------------------------------------------ K: forward/backward KLT
 * Replaces FeatureTracker::fbKltTracking(vprevpyr, vcurpyr, nwinsize, nbpyrlvl, ferr,
 * fmax_fbklt_dist, vkps, vpriorkps, vkpstatus) (/root/reference/src/feature_tracker.cpp:35-137;
 * declaration include/feature_tracker.hpp:44-47), i.e. forward cv::calcOpticalFlowPyrLK with
 * USE_INITIAL_FLOW|LK_GET_MIN_EIGENVALS, the status/err/inBorder filter, the level-0 backward
 * pass and the forward-backward distance test, fused per keypoint. */
typedef struct {
    int   win;        /* nwinsize (9) */
    int   max_iter;   /* klt_convg_crit_.maxCount (30) */
    float eps;        /* klt_convg_crit_.epsilon (0.01f) */
    float ferr;       /* nklt_err (30) */
    float fb_dist;    /* fmax_fbklt_dist (0.5) */
} ov2_klt_params;

/* n keypoints.  nbpyrlvl: per-keypoint pyramid depth (the reference's two calls, nbpyrlvl 1 for
 * keypoints with a 3D prior and 3 for the rest, visual_front_end.cpp:196,242, become one launch),
 * or NULL to use nbpyrlvl_all for every keypoint.  kps = vkps (n x 2 float), priors_inout =
 * vpriorkps (in: initial guess, out: forward result), status_out = vkpstatus (n bytes, 0/1).
 * Keypoints with x < 0 are empty-slot markers of fixed-stride batches (the detectors pad with (-1, -1)):
 * status 0, prior untouched. */
OV2_API ov2_status ov2_fb_klt(ov2_ctx* ctx, const ov2_pyr* prev, const ov2_pyr* cur, const ov2_klt_params* prm,
                      int n, const int32_t* frame_idx, int first_frame, int per_frame,
                      const uint8_t* nbpyrlvl, int nbpyrlvl_all,
                      const float* kps, float* priors_inout, uint8_t* status_out);

/* ------------------------------------------------------------------ F + S: grid FAST + cornerSubPix
 * Replaces FeatureExtractor::detectGridFAST(im, ncellsize, vcurkps, roi)
 * (/root/reference/src/feature_extractor.cpp:443-570; include/feature_extractor.hpp:41-42) with
 * the sequential ascending cell order as the defined semantics, including the CV_32F-mask byte
 * aliasing, libstdc++ std::sort tie resolution, the response >= 20 rule, disc painting, the
 * adaptive nfast_th_ update (:546-552) and cv::cornerSubPix((3,3),(-1,-1),{30,0.01}) (:556-565).
 *
 * Frames [first, first+count) of `pyr` (level 0).  Existing keypoints of frame k are
 * curkps[2*curkp_offsets[k] .. 2*curkp_offsets[k+1]) (curkp_offsets has count+1 entries; NULL =
 * no existing keypoints).  fast_th_inout[k] is the per-stream nfast_th_ state (in: threshold to
 * use, out: adapted threshold).  out_pts holds count * max_per_frame points (x, y float; unused
 * slots are set to (-1, -1)), in the reference's cell order; out_counts[k] = number found;
 * max_per_frame >= (H/cellsize)*(W/cellsize).  out_pts_int (optional, may be NULL) receives the
 * integer pixel positions before sub-pixel refinement (int32 x, y). */
OV2_API ov2_status ov2_grid_fast(ov2_ctx* ctx, const ov2_pyr* pyr, int first, int count, int cellsize,
                         const int32_t* curkp_offsets, const float* curkps,
                         int32_t* fast_th_inout, int max_per_frame,
                         float* out_pts, int32_t* out_counts, int32_t* out_pts_int, int do_subpix);

/* ------------------------------------------------------------------ D + S: single-scale detector + cornerSubPix
 * ("next" row, SURVEY.md 8f-1; the detector of the accurate/ and average/ configurations)
 * Replaces FeatureExtractor::detectSingleScale(im, ncellsize, vcurkps, roi)
 * (/root/reference/src/feature_extractor.cpp:288-440; include/feature_extractor.hpp:38-39): per cell
 * cv::GaussianBlur(3x3) + cv::cornerMinEigenVal(3, 3), first maximum of response * mask twice with the
 * disc mask, second detections admitted while cells stayed empty (:400-412), the adaptive dmaxquality_
 * update (:418-423) and cv::cornerSubPix (:424-436); sequential ascending cell order as the defined
 * semantics.  Arguments as ov2_grid_fast; roi_xywh = {x, y, width, height} on the HOST (NULL = whole
 * image); quality_inout[k] is the per-stream dmaxquality_ state (double, in/out); cellsize in [8, 64]. */
OV2_API ov2_status ov2_detect_single_scale(ov2_ctx* ctx, const ov2_pyr* pyr, int first, int count, int cellsize,
                         const int32_t* curkp_offsets, const float* curkps, const int32_t* roi_xywh,
                         double* quality_inout, int max_per_frame,
                         float* out_pts, int32_t* out_counts, int32_t* out_pts_int, int do_subpix);

/* Test hook: stage F1 alone (per-cell FAST-9/16 + NMS candidates of one frame, pre-filtered by the
 * mask byte rule), for cell-by-cell parity against cv::FastFeatureDetector. */
OV2_API ov2_status ov2_debug_fast_cells(ov2_ctx* ctx, const ov2_pyr* pyr, int frame, int cellsize, int fast_th,
                                uint32_t* cand_out, int32_t* cand_n_out, int cap_in, int* cap_out);

/* ------------------------------------------------------------------ ceresPnP (motion-only BA), "next" row 2
 * Replaces MultiViewGeometry::ceresPnP(vunkps, vwpts, vscales, Twc, nmaxiter, chi2th, buse_robust,
 * bapply_l2_after_robust, fx, fy, cx, cy, voutliersidx)
 * (/root/reference/src/multi_view_geometry.cpp:492-588; called per frame at src/visual_front_end.cpp:791-801),
 * batched: problem k owns points [offsets[k], offsets[k+1]) of unpx ([N][2] undistorted pixels), wpts ([N][3]
 * world points) and scales (pyramid level per point or NULL), calibration K[k] = fx, fy, cx, cy and pose
 * Twc[k] = tx,ty,tz,qx,qy,qz,qw (in: initial guess, out: refined; unchanged when every block is rejected).
 * ReprojectionErrorSE3 residuals with SE3LeftParameterization, HuberLoss(sqrt(chi2th)), Ceres' Levenberg-
 * Marquardt loop (DENSE_QR in the reference; 6x6 damped normal equations here), max nmaxiter iterations,
 * function tolerance 1e-3; blocks with chi2 > chi2th or non-positive depth after the first solve are flagged
 * in outlier_flags (and removed before an L2 re-solve when apply_l2_after_robust).  success_out[k] = the
 * reference's return value.  The 5 ms wall-clock cap of the reference (:538) is not modelled.
 * offsets must be a HOST pointer; iterations_out (optional) = LM iterations of the last solve of each problem.
 * STATUS (round 1): validated on the host against the oracle; not yet run on a B200. */
OV2_API ov2_status ov2_pnp_solve(ov2_ctx* ctx, int nprob, const int32_t* offsets, const double* unpx, const double* wpts,
                         const int32_t* scales, const double* K, double* pose_inout, int nmaxiter, float chi2th,
                         int use_robust, int apply_l2_after_robust, uint8_t* outlier_flags, uint8_t* success_out,
                         int32_t* iterations_out);

/* ------------------------------------------------------------------ B: descriptors
 * Replaces FeatureExtractor::describeBRIEF(im, vpts)
 * (/root/reference/src/feature_extractor.cpp:224-285), non-contrib branch
 * cv::ORB::create(500, 1., 0) (:245): 256 tests of the ORB pattern on the float32-Gaussian
 * smoothed image, centre = cvRound(pt), points whose rounded centre is closer than 31 px to the
 * border (and points with x < 0, used as "empty slot" markers) get valid = 0 and a zero
 * descriptor, mirroring the empty cv::Mat the reference returns for them. */
OV2_API ov2_status ov2_describe(ov2_ctx* ctx, const ov2_pyr* pyr, int n, const int32_t* frame_idx, int first_frame, int per_frame,
                        const float* pts, uint8_t* desc32_out, uint8_t* valid_out);

/* Descriptor selection for ov2_describe on this context (the reference selects it at compile time,
 * /root/reference/CMakeLists.txt:12,35-39 and src/feature_extractor.cpp:69-70,242-246):
 *   OV2_DESC_ORB_FALLBACK (default, pairs = NULL): the non-contrib branch described above.
 *   OV2_DESC_BRIEF32: cv::xfeatures2d::BriefDescriptorExtractor::create() (32 bytes, no orientation):
 *     256 tests SMOOTHED(y0, x0) < SMOOTHED(y1, x1) of 9 x 9 box sums around (int)(pt + 0.5), first test of a
 *     byte in bit 7, border 28 px.  `pairs` = int8[256][4] = (y0, x0, y1, x1) in the order of opencv_contrib's
 *     modules/xfeatures2d/src/generated_32.i (that table is not redistributed here; |offset| <= 24 is checked). */
#define OV2_DESC_ORB_FALLBACK 0
#define OV2_DESC_BRIEF32 1
OV2_API ov2_status ov2_describe_config(ov2_ctx* ctx, int mode, const int8_t* pairs);

/* ------------------------------------------------------------------ 8f-3: stereo prior by a row search
 * Replaces the per-keypoint loop over FeatureTracker::getLineMinSAD(iml, imr, pt, nwinsize, xprior, l1err, bgoleft)
 * (/root/reference/src/feature_tracker.cpp:138-204) that MapManager::stereoMatching runs for every 2-D keypoint of a
 * keyframe on the coarsest pyramid level when `bdo_stereo_rect` is set (/root/reference/src/map_manager.cpp:417-431):
 * for each point (coordinates of pyramid level `level`) the column of the right image, scanned in unit steps from the
 * point's own column (downwards when goleft), whose nwinsize x nwinsize window has the smallest mean absolute
 * difference to the sub-pixel patch of the left image.  xprior_out = that column (float, same fractional part as the
 * input) or -1 when the window shrinks to nothing at the border / no candidate is below 255; l1err_out = the minimum
 * (255 when xprior is -1; the reference leaves it unset there).  nwinsize must be odd (OV2_ERR_INVALID otherwise, the
 * reference prints a message and returns) and <= 15.  Frame addressing as ov2_fb_klt. */
OV2_API ov2_status ov2_line_min_sad(ov2_ctx* ctx, const ov2_pyr* left, const ov2_pyr* right, int level, int n,
                            const int32_t* frame_idx, int first_frame, int per_frame, const float* pts, int nwinsize,
                            int goleft, float* xprior_out, float* l1err_out);

/* ------------------------------------------------------------------ 8f-4: local-map matching
 * The data-parallel core of Mapper::matchToMap(frame, fmaxprojerr, fdistratio, set_local_lmids)
 * (/root/reference/src/mapper.cpp:576-774): for every candidate map point of the local map (cand_mp, in the caller's
 * iteration order) projection into the frame, culling, the keypoints of the four surrounding grid cells
 * (Frame::getSurroundingKeypoints, src/frame.cpp:624-650), pixel distance, "never observed together", mean co-projection
 * error, minimal descriptor distance (MapPoint::computeMinDescDist, src/map_point.cpp:236-252), best / second with the
 * 0.9 ratio test -> best_kp_out[ncand] (keypoint index or -1), best_dist_out[ncand]; then per keypoint the candidate with
 * the smallest distance (later candidates win ties) -> kp_match_out[nkps] (index INTO cand_mp or -1), kp_dist_out[nkps]
 * (1024 when unmatched).  The caller (the Mapper shim) flattens the map and applies the merges (mapper.cpp:559-570).
 * Map-point table = the candidates AND the map points of the frame's keypoints.  Rotations are 3x3 matrices (row major)
 * followed by the translation: Tcw[12], kf_Tcw[nkfs][12].  dist = (k1, k2, p1, p2, k3) of the pinhole model or NULL
 * (fisheye calibrations are not built: keep the reference's matchToMap for them).  dmaxpxdist = fmaxprojerr, doubled by
 * the caller when the frame has fewer than 30 3-D keypoints (:597-600); view_th = cos(max half field of view) (:586-596). */
typedef struct {
    double Tcw[12]; double K[4]; const double* dist;
    int img_w, img_h, ncellsize, nbwcells, ncells;
    const int32_t* cell_ptr;      /* [ncells + 1] keypoints per grid cell (Frame::vgridkps_), CSR */
    const int32_t* cell_kp;       /* [nkps] keypoint indices, cell by cell, in the cell lists' order */
    int nkps; const float* kp_px; /* [nkps][2] kp.px_ */
    const int32_t* kp_lm;         /* [nkps] map-point table index of the keypoint's map point, -1: none */
    int nmps; const double* mp_xyz;                                   /* [nmps][3] */
    const int32_t* mp_desc_ptr; int ndesc; const uint8_t* desc;       /* [nmps + 1], [ndesc][32] */
    const uint64_t* mp_kfmask;    /* [nmps][4] bit k: observed by local keyframe k (k < 256) */
    const int32_t* mp_obs_ptr; int nobs; const int32_t* obs_kf; const float* obs_px;   /* [nmps + 1], [nobs], [nobs][2] */
    int nkfs; const double* kf_Tcw;                                   /* [nkfs][12] */
    int ncand; const int32_t* cand_mp;
    float dmaxpxdist, fdistratio, view_th;
} ov2_match_problem;
OV2_API ov2_status ov2_match_to_map(ov2_ctx* ctx, const ov2_match_problem* p, int32_t* best_kp_out, float* best_dist_out,
                            int32_t* kp_match_out, float* kp_dist_out);

/* ------------------------------------------------------------------ composite: one front-end step
 * P(prev), P(cur), K, F+S on cur (no existing keypoints), B(tracked), B(new) for `count` frame pairs in
 * ONE call (batch mode inside): what VisualFrontEnd::trackMono + MapManager::extractKeypoints do per
 * frame (/root/reference/src/visual_front_end.cpp:65-128, src/map_manager.cpp:286-341).  Pointers
 * host or device as everywhere; n_kps = count * kps_per_frame; cellsize <= 0 skips F/B(new).
 * The step is captured into a CUDA graph per distinct argument block (at most 16 are kept per context): zero the struct
 * before filling it (its padding bytes are part of the cache key), and reuse argument blocks - a block that changes every
 * call runs eagerly.  A detector cell that exceeds its candidate capacity makes the call return OV2_ERR_CAPACITY. */
typedef struct {
    const uint8_t* prev_images; const uint8_t* cur_images; size_t row_stride, frame_stride; int count;
    ov2_klt_params klt; int n_kps, kps_per_frame; const uint8_t* nbpyrlvl; int nbpyrlvl_all;
    const float* kps; float* priors_inout; uint8_t* status_out;
    int cellsize; int32_t* fast_th_inout; int max_per_frame; float* new_pts; int32_t* new_counts;
    uint8_t* desc_tracked; uint8_t* valid_tracked; uint8_t* desc_new; uint8_t* valid_new;
} ov2_frontend_step_args;
OV2_API ov2_status ov2_frontend_step(ov2_ctx* ctx, ov2_pyr* prev, ov2_pyr* cur, const ov2_frontend_step_args* args);

/* ------------------------------------------------------------------ L: local bundle adjustment
 * Replaces the solve sections of Optimizer::localBA(Frame&, bool)
 * (/root/reference/src/optimizer.cpp:436-479 robust solve, :492-594 outlier scan,
 *  :603-627 refinement, :637-735 second scan), i.e. Ceres 2.0 TrustRegionMinimizer +
 * LevenbergMarquardtStrategy + SCHUR linear solver on ReprojectionErrorKSE3AnchInvDepth
 * residuals (src/ceres_parametrization.cpp:361-473) with SE3LeftParameterization.
 * The flat problem description is what localBA's setup (:43-430) builds from the map. */
typedef struct {
    int32_t  ncam, npts, nobs;
    const double*  K;              /* [4] fx, fy, cx, cy (constant block) */
    double*        pose;           /* [ncam][7] Twc = tx,ty,tz,qx,qy,qz,qw ; in/out */
    const uint8_t* pose_const;     /* [ncam] 1 = SetParameterBlockConstant */
    const int32_t* lm_anchor_cam;  /* [npts] */
    const double*  lm_anchor_px;   /* [npts][2] undistorted anchor pixel */
    double*        lm_invdepth;    /* [npts] in/out */
    const int32_t* obs_cam;        /* [nobs] observing camera (non-anchor observations) */
    const int32_t* obs_lm;         /* [nobs] landmark index, sorted ascending (CSR by landmark) */
    const double*  obs_px;         /* [nobs][2] */
    /* stereo windows (NULL / ignored for mono): residual type per observation -
     *   0 left camera, other keyframe    ReprojectionErrorKSE3AnchInvDepth             (ceres_parametrization.cpp:361-473)
     *   1 right camera, other keyframe   ReprojectionErrorRightCamKSE3AnchInvDepth     (:579-712)
     *   2 right camera, anchor keyframe  ReprojectionErrorRightAnchCamKSE3AnchInvDepth (:476-577; obs_cam = anchor)
     * Kr = right calibration [4], Trl = constant right-from-left extrinsic [7] (tx..tz, qx..qw). */
    const uint8_t* obs_type;       /* [nobs] or NULL */
    const double*  Kr;             /* [4] or NULL */
    const double*  Trl;            /* [7] or NULL */
} ov2_ba_problem;

typedef struct {
    int    max_iters_robust;   /* 5  (optimizer.cpp:462) */
    int    max_iters_refine;   /* 10 (optimizer.cpp:610) */
    double huber_th;           /* robust_mono_th = 5.9915 (loss = HuberLoss(sqrt(th)), :49) */
    double function_tolerance; /* 1e-3 (:463) */
    int    use_robust;         /* buse_robust_cost */
    int    apply_l2_after_robust; /* (:603) */
    int    refine_loss;        /* refinement loss: -1 = as the reference decides (trivial loss iff left-camera AND
                                * other-frame right-camera residuals both survive the first scan, :606-608; i.e.
                                * mono windows keep Huber), 0 = keep the robust loss, 1 = trivial loss */
} ov2_ba_opts;

typedef struct {
    int    iters_robust, iters_refine;  /* LM iterations executed (successful + unsuccessful) */
    double initial_cost, final_cost;    /* of the last solve that ran */
    int    n_outliers_first, n_outliers_second;
    int    termination;                 /* 0 convergence, 1 max iterations, 2 failure */
} ov2_ba_result;

/* Capacity of one ov2_localba_solve window (the loop closer's looseBA and fullBA hand over windows of hundreds of
 * keyframes).  Windows of up to OV2_BA_SMALL_MAX_OPT_KEYFRAMES optimised keyframes run the kernel of csrc/ba_lm.cu (or, with
 * more than OV2_BA_SMALL_MAX_KEYFRAMES keyframes in total, the round-1 path, which has no limit on the total); larger ones the
 * large-window kernel of csrc/ba_large.cu, whose dense tiled reduced system needs (6 x optimised keyframes)^2 x 8 bytes
 * (302 MB at the cap) besides ~310 bytes per residual block; a window whose device memory plan exceeds
 * OV2_BA_LARGE_MAX_BYTES is refused with OV2_ERR_CAPACITY.  ov2_localba_solve_batch, _p2p and _sharded keep the small-window
 * limits. */
#define OV2_BA_MAX_OPT_KEYFRAMES       1024
#define OV2_BA_MAX_KEYFRAMES           4096
#define OV2_BA_SMALL_MAX_OPT_KEYFRAMES 64
#define OV2_BA_SMALL_MAX_KEYFRAMES     256
#define OV2_BA_LARGE_MAX_BYTES         (16ull << 30)

/* outlier_out (optional): [nobs] bytes, bit0 = flagged after solve #1, bit1 = after solve #2.
 * The whole two-stage solve (both Ceres solves, every LM iteration, both outlier scans) is ONE kernel launch with the
 * trust-region controller on the device (csrc/ba_lm.cu, csrc/ba_large.cu); OV2_BA_LEGACY=1 selects the round-1 path (one
 * launch per phase, controller on the host, at most 64 optimised keyframes) as a cross-check.  At most
 * OV2_BA_MAX_OPT_KEYFRAMES optimised and OV2_BA_MAX_KEYFRAMES total keyframes per window (more: OV2_ERR_CAPACITY), or
 * at most OV2_BA_SMALL_MAX_OPT_KEYFRAMES optimised keyframes and any total.
 * Residency of a window's arrays is decided on `pose`: host poses = every array of the window (and outlier_out) is host
 * memory, the reference's flow; device poses = each array is inspected and may be either. */
OV2_API ov2_status ov2_localba_solve(ov2_ctx* ctx, const ov2_ba_problem* pb, const ov2_ba_opts* opts,
                             ov2_ba_result* res, uint8_t* outlier_out);

/* K independent windows in ONE launch (the solves/s metric; SURVEY.md 7 "hard parts" (ii)), each of at most 64 optimised and
 * 256 total keyframes (more: OV2_ERR_CAPACITY): window k is pbs[k] with results[k]
 * and outlier_outs[k] (NULL entries / NULL array allowed); the same options for every window.  Groups of thread blocks pull
 * windows round-robin, every group runs the whole two-stage solve of its window on the device. */
OV2_API ov2_status ov2_localba_solve_batch(ov2_ctx* ctx, int nprob, const ov2_ba_problem* pbs, const ov2_ba_opts* opts,
                                   ov2_ba_result* results, uint8_t* const* outlier_outs);

/* Optimizer::signalStopLocalBA / stopLocalBA (/root/reference/src/optimizer.cpp:2334-2343, raised by Estimator::addNewKf,
 * src/estimator.cpp:228-232): stop = 1 asks the solve running (or about to run) on `ctx` to skip the L2 refinement; the
 * solve kernel polls the flag where the reference does (optimizer.cpp:603-604).  May be called from another host thread
 * while ov2_localba_solve runs; the caller clears it (stop = 0) as optimizer.cpp:896 does. */
OV2_API ov2_status ov2_localba_request_stop(ov2_ctx* ctx, int stop);

/* Multi-GPU localBA over PEER MEMORY (BASELINE.json configs[4], SURVEY.md 8e).  One process per GPU (or several contexts in one
 * process): every rank creates a communicator (it allocates the rank's exchange buffer), the 64-byte CUDA IPC handles are
 * exchanged by the caller (torch.distributed.all_gather, MPI, a pipe ...) and handed to ov2_ba_comm_connect.  The solve is
 * collective: every rank calls ov2_localba_solve_p2p with ITS shard (landmarks with all their observations partitioned over
 * the ranks, every rank holds all keyframe poses; a shard may be empty).  Inside the solve kernel every LM iteration sums
 * the ranks' partial reduced camera systems [cost, rhs, F'r, column norms, S] straight out of peer memory over NVLink
 * (rank order, so every rank holds bit-identical sums, solves the same system and takes the same decisions): no NCCL call
 * and no host round trip between iterations.  Poses come back identical on all ranks, inverse depths / flags / outlier
 * counts are the shard's own. */
typedef struct ov2_ba_comm ov2_ba_comm;
OV2_API ov2_status ov2_ba_comm_create(ov2_ctx* ctx, int rank, int world, ov2_ba_comm** out);       /* world <= 8 */
OV2_API ov2_status ov2_ba_comm_handle(ov2_ba_comm* comm, void* handle_out, size_t handle_bytes);    /* >= 64 bytes */
OV2_API ov2_status ov2_ba_comm_connect(ov2_ba_comm* comm, const void* handles, size_t handle_stride);   /* world handles, rank order */
OV2_API ov2_status ov2_ba_comm_connect_local(ov2_ba_comm* comm, ov2_ba_comm* const* all);            /* all ranks in this process */
OV2_API void       ov2_ba_comm_destroy(ov2_ba_comm* comm);
OV2_API ov2_status ov2_localba_solve_p2p(ov2_ctx* ctx, ov2_ba_comm* comm, const ov2_ba_problem* pb, const ov2_ba_opts* opts,
                                 ov2_ba_result* res, uint8_t* outlier_out);

/* Multi-GPU localBA, callback variant (round 1; the collective is whatever the caller wires in, e.g. ncclAllReduce):
 * landmarks (with all their observations) are
 * partitioned over ranks, every rank holds all keyframe poses.  `pb` describes THIS rank's shard
 * (ncam / pose / pose_const identical on all ranks; npts / nobs local, may be 0 observations).
 * Per LM iteration the partial reduced camera system [cost, rhs, F'r, column norms, S] is summed
 * over ranks by ONE call of `allreduce` (the caller wires it to ncclAllReduce / torch.distributed
 * over NVLink), followed by a 4-double collective for the candidate cost and model decrease; all
 * ranks then solve the same reduced system and take identical LM decisions (no broadcast).
 * allreduce(user, device_buf, count, cuda_stream): in-place SUM of `count` doubles on the given
 * stream (or synchronously); returns 0 on success.  Result counts (outliers) are per shard. */
typedef int (*ov2_allreduce_fn)(void* user, double* device_buf, size_t count, void* cuda_stream);
OV2_API ov2_status ov2_localba_solve_sharded(ov2_ctx* ctx, const ov2_ba_problem* pb, const ov2_ba_opts* opts,
                                     ov2_ba_result* res, uint8_t* outlier_out, ov2_allreduce_fn allreduce,
                                     void* user, int rank);

#ifdef __cplusplus
}
#endif
#endif /* OV2B200_H */
