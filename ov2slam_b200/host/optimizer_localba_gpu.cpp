// Optimizer::localBA on the GPU: the reference's declaration (include/optimizer.hpp:33-67) is kept,
// this translation unit supplies Optimizer::localBA(Frame&, bool) so estimator.cpp:91 links
// unchanged; the other Optimizer members (looseBA, fullBA, pose graphs, stop flags) stay in the
// reference's own optimizer.cpp built with -DOV2_EXTERNAL_LOCALBA (one #ifndef around its localBA
// body, see INTEGRATION.md).
//
// Compile-checked and self-tested in this container against stand-in headers that mirror the reference's class
// interfaces (host/standin/ref/: optimizer.hpp, map_manager.hpp, sophus/se3.hpp, Eigen/Dense) - the reference's own
// headers need ROS, PCL, OpenCV, Eigen and Sophus, none of which exist here (SURVEY.md section 0);
// host/optimizer_selftest.cpp builds a synthetic map, runs this localBA and tests/test_host_shim.py compares the
// map it leaves behind with the flat solve of the same window.  On a box that builds the reference, compile this file
// with the reference's include path instead of the stand-ins.
// Mono and stereo windows (inverse-depth parametrisation, buse_inv_depth_ = 1: every shipped
// configuration); the XYZ parametrisation (buse_inv_depth_ = 0) is not flattened and falls through
// with a diagnostic.
//
// What stays on the host is exactly the part SURVEY.md 8a row G scopes out of acceleration: walking
// the covisibility graph / hash maps to FLATTEN the window into the SoA arrays ov2_localba_solve
// takes, and applying the result to the map.  The numerical work (Ceres in the reference,
// optimizer.cpp:436-735) is one ABI call = one kernel launch.
#include <atomic>
#include <chrono>
#include <iostream>
#include <algorithm>
#include <map>
#include <set>
#include <thread>
#include <unordered_map>
#include <vector>

#include <unordered_set>

#include "optimizer.hpp"          // the reference's, unchanged
#include "../../include/ov2b200.h"

namespace {

ov2_ctx* ba_context() {
    static ov2_ctx* ctx = nullptr;                   // estimator thread only (optim_mutex_, estimator.cpp:85)
    if (!ctx && ov2_create(0, &ctx) != OV2_OK) ctx = nullptr;
    return ctx;
}

// Flat window: camera index <-> keyframe id, landmark index <-> map point id.
struct Window {
    std::vector<int> kfids;  std::unordered_map<int, int> cam_of_kf;
    std::vector<std::shared_ptr<Frame>> kfs;
    std::vector<double> pose;  std::vector<uint8_t> pose_const;
    std::vector<int> lmids;  std::vector<std::shared_ptr<MapPoint>> lms;
    std::vector<int32_t> lm_anchor_cam;  std::vector<double> lm_anchor_px, lm_invdepth;
    std::vector<int32_t> obs_cam, obs_lm;  std::vector<double> obs_px;  std::vector<uint8_t> obs_type;

    // residual type as include/ov2b200.h: 0 left camera / other keyframe, 1 right camera / other keyframe,
    // 2 right camera / anchor keyframe (obs_cam = anchor)
    void add_obs(int cam, int lm, double u, double v, uint8_t type) {
        obs_cam.push_back(cam); obs_lm.push_back(lm); obs_px.push_back(u); obs_px.push_back(v); obs_type.push_back(type);
    }

    int add_camera(int kfid, const std::shared_ptr<Frame>& kf, bool constant) {
        auto it = cam_of_kf.find(kfid);
        if (it != cam_of_kf.end()) return it->second;
        const int c = (int)kfids.size();
        cam_of_kf.emplace(kfid, c);
        kfids.push_back(kfid);
        kfs.push_back(kf);
        const Sophus::SE3d T = kf->getTwc();
        const Eigen::Quaterniond q = T.unit_quaternion();
        const Eigen::Vector3d t = T.translation();
        const double p[7] = {t.x(), t.y(), t.z(), q.x(), q.y(), q.z(), q.w()};   // se3_param_block.hpp:39-46
        pose.insert(pose.end(), p, p + 7);
        pose_const.push_back(constant ? 1 : 0);
        return c;
    }
};


// Landmarks of the window: the first valid observer (ascending keyframe id) anchors the inverse depth, every further observer
// contributes one residual block (two for a stereo keypoint); observers outside the window join it as constant keyframes.
// The same loop body in localBA (optimizer.cpp:191-392), looseBA (:1023-1226) and fullBA (:1794-1990).
void flatten_landmarks(MapManager& map, Window& win, const std::vector<int>& lm_order, const int newest, const bool stereo) {
    MapManager* pmap_ = &map;
    for (int lmid : lm_order) {
        auto lm = pmap_->getMapPoint(lmid);
        if (!lm || lm->isBad()) continue;
        int anchor_cam = -1;
        const int l = (int)win.lmids.size();
        for (int kfid : lm->getKfObsSet()) {
            if (kfid > newest) continue;
            auto cit = win.cam_of_kf.find(kfid);
            std::shared_ptr<Frame> kf = cit != win.cam_of_kf.end() ? win.kfs[cit->second] : pmap_->getKeyframe(kfid);
            if (!kf) { pmap_->removeMapPointObs(kfid, lmid); continue; }
            const int cam = win.add_camera(kfid, kf, /*constant=*/cit == win.cam_of_kf.end());
            const auto kp = kf->getKeypointById(lmid);
            if (kp.lmid_ != lmid) { pmap_->removeMapPointObs(lmid, kfid); continue; }
            // kp.scale_ is 0 for every keypoint the reference's front-end creates (map_manager.cpp adds
            // keypoints without a scale), so the residuals' information matrix 2^-scale * I is the identity
            if (anchor_cam < 0) {
                anchor_cam = cam;
                win.lmids.push_back(lmid);
                win.lms.push_back(lm);
                win.lm_anchor_cam.push_back(cam);
                win.lm_anchor_px.push_back(kp.unpx_.x);
                win.lm_anchor_px.push_back(kp.unpx_.y);
                win.lm_invdepth.push_back(1.0 / (kf->getTcw() * lm->getPoint()).z());
                // the anchor's own right-camera observation constrains the inverse depth alone (optimizer.cpp:268-284)
                if (stereo && kp.is_stereo_) win.add_obs(cam, l, kp.runpx_.x, kp.runpx_.y, 2);
                continue;
            }
            win.add_obs(cam, l, kp.unpx_.x, kp.unpx_.y, 0);            // appended landmark by landmark: already sorted
            if (stereo && kp.is_stereo_) win.add_obs(cam, l, kp.runpx_.x, kp.runpx_.y, 1);   // (optimizer.cpp:295-324)
        }
    }
}

// Gauge (at least two constant keyframes in mono, one in stereo: optimizer.cpp:65-69, 396-407 / :1228-1239 / :1992-2003) and the solver's
// capacity (OV2_BA_MAX_OPT_KEYFRAMES optimised keyframes: beyond that the OLDEST optimised keyframes are held constant, said once
// on stderr).  A window of more than OV2_BA_MAX_KEYFRAMES keyframes in total (a fullBA over a very long run) cannot take the
// large-window solve at all, whatever is held constant: it keeps OV2_BA_SMALL_MAX_OPT_KEYFRAMES (64) optimised keyframes, the
// window the round-1 solve takes at any total size.
// `reference_walk` (localBA): the reference walks its keyframe hash map from begin() and counts every keyframe it visits, constant
// already or not (`nbcstkfs++`, :400-406) - with libstdc++ the walk starts at the LAST keyframe inserted, which is keyframe 0 of a
// fully covisible window: it is "fixed" a second time, the count reaches two and only ONE keyframe is constant.  The drop-in does the
// same walk over a hash map filled in the same order (Window::cam_of_kf), so that it fixes what the reference fixes
// (tests/test_oracle_vs_reference_map.py runs the reference's own localBA next to it).  looseBA / fullBA keep ascending keyframe ids.
void fix_gauge_and_capacity(Window& win, const bool stereo, const char* who, const bool reference_walk = false) {
    size_t nconst = 0;
    for (uint8_t c : win.pose_const) nconst += c;
    const size_t nmincst = stereo ? 1 : 2;
    std::map<int, int> by_id(win.cam_of_kf.begin(), win.cam_of_kf.end());
    if (reference_walk) {
        for (auto it = win.cam_of_kf.begin(); nconst < nmincst && it != win.cam_of_kf.end(); ++it) { win.pose_const[it->second] = 1; nconst++; }
        nconst = 0;
        for (uint8_t c : win.pose_const) nconst += c;
    } else {
        for (auto it = by_id.begin(); nconst < nmincst && it != by_id.end(); ++it)
            if (!win.pose_const[it->second]) { win.pose_const[it->second] = 1; nconst++; }
    }
    size_t nvar = win.pose_const.size() - nconst;
    const size_t cap = win.pose_const.size() > OV2_BA_MAX_KEYFRAMES ? OV2_BA_SMALL_MAX_OPT_KEYFRAMES : OV2_BA_MAX_OPT_KEYFRAMES;
    if (nvar > cap) {
        static bool told = false;
        if (!told) { std::cerr << "[ov2b200] " << who << ": " << nvar << " optimised keyframes, the oldest " << nvar - cap << " are held constant\n"; told = true; }
        for (auto it = by_id.begin(); nvar > cap && it != by_id.end(); ++it)
            if (!win.pose_const[it->second]) { win.pose_const[it->second] = 1; nvar--; }
    }
}

// ov2_ba_problem view of a window (K / Kr / Trl storage supplied by the caller).
void make_problem(const Window& win, Window& wmut, const Frame& ref, const bool stereo, double K[4], double Kr[4], double Trl[7], ov2_ba_problem& pb) {
    auto cal = ref.pcalib_leftcam_;
    K[0] = cal->fx_; K[1] = cal->fy_; K[2] = cal->cx_; K[3] = cal->cy_;
    pb.ncam = (int)win.kfids.size(); pb.npts = (int)win.lmids.size(); pb.nobs = (int)win.obs_cam.size();
    pb.K = K; pb.pose = wmut.pose.data(); pb.pose_const = win.pose_const.data();
    pb.lm_anchor_cam = win.lm_anchor_cam.data(); pb.lm_anchor_px = win.lm_anchor_px.data();
    pb.lm_invdepth = wmut.lm_invdepth.data();
    pb.obs_cam = win.obs_cam.data(); pb.obs_lm = win.obs_lm.data(); pb.obs_px = win.obs_px.data();
    pb.obs_type = nullptr; pb.Kr = nullptr; pb.Trl = nullptr;
    if (stereo) {
        auto calr = ref.pcalib_rightcam_;
        Kr[0] = calr->fx_; Kr[1] = calr->fy_; Kr[2] = calr->cx_; Kr[3] = calr->cy_;
        const Sophus::SE3d T = calr->getExtrinsic().inverse();          // Trl (optimizer.cpp:112-114)
        const Eigen::Quaterniond q = T.unit_quaternion();
        const Eigen::Vector3d t = T.translation();
        const double e[7] = {t.x(), t.y(), t.z(), q.x(), q.y(), q.z(), q.w()};
        for (int i = 0; i < 7; ++i) Trl[i] = e[i];
        pb.obs_type = win.obs_type.data(); pb.Kr = Kr; pb.Trl = Trl;
    }
}

}  // namespace

void Optimizer::localBA(Frame &newframe, const bool buse_robust_cost)
{
    // Early-outs of the reference (optimizer.cpp:61-63): poor tracking -> no BA.
    const int nmincov = pslamstate_->nmin_covscore_;
    if ((int)newframe.nb3dkps_ < nmincov) return;
    ov2_ctx* ctx = ba_context();
    if (!ctx) { std::cerr << "[ov2b200] localBA: no CUDA device (no CPU fallback)\n"; return; }
    const bool stereo = pslamstate_->stereo_;
    if (!pslamstate_->buse_inv_depth_) {
        std::cerr << "[ov2b200] localBA: only the anchored inverse-depth parametrisation (buse_inv_depth: 1) is built\n";
        return;
    }

    // ---- 1. window: covisible keyframes, newest first; optimise while the covisibility score holds,
    //         everything older than the first weak keyframe is constant (optimizer.cpp:128-188)
    Window win;
    std::map<int, int> cov = newframe.getCovisibleKfMap();
    cov.emplace(newframe.kfid_, newframe.nb3dkps_);
    std::unordered_set<int> set_lmids2opt;   // landmark ids seen from optimised keyframes; walked in the hash set's order, as the reference
    bool freeze = false;                     // does (:135, :191): it decides in which order keyframes outside the window join it
    const int newest = cov.rbegin()->first;
    for (auto it = cov.rbegin(); it != cov.rend(); ++it) {
        const int kfid = it->first;
        const int score = kfid > newframe.kfid_ ? (int)newframe.nbkps_ : it->second;
        auto kf = pmap_->getKeyframe(kfid);
        if (!kf) { newframe.removeCovisibleKf(kfid); continue; }
        const bool optimise = score >= nmincov && !freeze && kfid > 0;
        if (!optimise) freeze = true;
        win.add_camera(kfid, kf, !optimise);
        if (optimise)
            for (const auto& kp : kf->getKeypoints3d()) set_lmids2opt.insert(kp.lmid_);
    }

    // ---- 2. landmarks (optimizer.cpp:191-392)
    const std::vector<int> lm_order(set_lmids2opt.begin(), set_lmids2opt.end());
    flatten_landmarks(*pmap_, win, lm_order, newest, stereo);
    // ---- 3. gauge + solver capacity
    fix_gauge_and_capacity(win, stereo, "localBA", /*reference_walk=*/true);
    if (win.obs_cam.empty()) return;

    // ---- 4. solve on the GPU (replaces ceres::Solve x2 + the two outlier scans)
    double K[4], Kr[4] = {0, 0, 0, 0}, Trl[7] = {0, 0, 0, 0, 0, 0, 1};
    ov2_ba_problem pb;
    make_problem(win, win, newframe, stereo, K, Kr, Trl, pb);
    ov2_ba_opts op;
    op.max_iters_robust = 5; op.max_iters_refine = 10;                // optimizer.cpp:462, :610
    op.huber_th = pslamstate_->robust_mono_th_; op.function_tolerance = 1.e-3;
    op.use_robust = buse_robust_cost ? 1 : 0;
    op.apply_l2_after_robust = pslamstate_->apply_l2_after_robust_ ? 1 : 0;
    op.refine_loss = -1;                                              // as optimizer.cpp:606-608 decides
    ov2_ba_result res;
    std::vector<uint8_t> flags(win.obs_cam.size(), 0);
    // The reference polls stopLocalBA() once, between the robust solve and the refinement (optimizer.cpp:603-604); the
    // stop request arrives from the mapper thread (estimator.cpp:228-232) while the solve is running.  The solve kernel
    // polls a flag at exactly that point (ov2_localba_request_stop); a watcher forwards bstop_localba_ to it, so the
    // reference's signalStopLocalBA() needs no edit.
    ov2_localba_request_stop(ctx, stopLocalBA() ? 1 : 0);
    std::atomic<bool> solve_done{false};
    std::thread watcher([&]() {
        while (!solve_done.load(std::memory_order_acquire)) {
            if (bstop_localba_) { ov2_localba_request_stop(ctx, 1); return; }
            std::this_thread::sleep_for(std::chrono::microseconds(20));
        }
    });
    const ov2_status solve_rc = ov2_localba_solve(ctx, &pb, &op, &res, flags.data());
    solve_done.store(true, std::memory_order_release);
    watcher.join();
    ov2_localba_request_stop(ctx, 0);
    if (solve_rc != OV2_OK) {
        std::cerr << "[ov2b200] localBA: " << ov2_last_error(ctx) << "\n";
        bstop_localba_ = false;
        return;                                                        // map untouched
    }

    // ---- 5. apply to the map under map_mutex_ (optimizer.cpp:741-897)
    std::lock_guard<std::mutex> lock(pmap_->map_mutex_);
    std::unordered_map<int, int> suspicious;                           // lmid -> had a rejected observation
    // rejected right-camera observations only lose their stereo half (removeStereoKeypointById,
    // optimizer.cpp:742-750); rejected left-camera observations are removed from the map (:752-763)
    for (size_t i = 0; i < flags.size(); ++i) {
        if (!flags[i] || win.obs_type[i] == 0) continue;
        win.kfs[win.obs_cam[i]]->removeStereoKeypointById(win.lmids[win.obs_lm[i]]);
        suspicious.emplace(win.lmids[win.obs_lm[i]], 1);
    }
    for (size_t i = 0; i < flags.size(); ++i) {
        if (!flags[i] || win.obs_type[i] != 0) continue;
        const int kfid = win.kfids[win.obs_cam[i]], lmid = win.lmids[win.obs_lm[i]];
        pmap_->removeMapPointObs(lmid, kfid);
        if (kfid == pmap_->pcurframe_->kfid_) pmap_->removeObsFromCurFrameById(lmid);
        suspicious.emplace(lmid, 1);
    }
    for (size_t c = 0; c < win.kfids.size(); ++c) {
        if (win.pose_const[c]) continue;
        const double* p = &win.pose[7 * c];
        win.kfs[c]->setTwc(Sophus::SE3d(Eigen::Quaterniond(p[6], p[3], p[4], p[5]), Eigen::Vector3d(p[0], p[1], p[2])));
    }
    auto cull_if_weak = [&](int lmid, const std::shared_ptr<MapPoint>& lm) {
        if (lm->isBad()) { pmap_->removeMapPoint(lmid); return true; }
        if (lm->getKfObsSet().size() < 3 && lm->kfid_ < newframe.kfid_ - 3 && !lm->isobs_) { pmap_->removeMapPoint(lmid); return true; }
        return false;
    };
    for (size_t l = 0; l < win.lmids.size(); ++l) {
        const int lmid = win.lmids[l];
        auto lm = win.lms[l];
        if (cull_if_weak(lmid, lm)) { suspicious.erase(lmid); continue; }
        const double invd = win.lm_invdepth[l];
        if (1.0 / invd <= 0.0) { pmap_->removeMapPoint(lmid); suspicious.erase(lmid); continue; }
        auto ait = win.cam_of_kf.find(lm->kfid_);                       // anchor looked up by the map point's own kf id
        if (ait == win.cam_of_kf.end()) { suspicious.emplace(lmid, 1); continue; }
        auto kfa = win.kfs[ait->second];
        const auto kp = kfa->getKeypointById(lmid);
        const Eigen::Vector3d ray(kp.unpx_.x, kp.unpx_.y, 1.0);
        pmap_->updateMapPoint(lmid, kfa->getTwc() * ((1.0 / invd) * kfa->pcalib_leftcam_->iK_ * ray), invd);
    }
    for (const auto& s : suspicious) {
        auto lm = pmap_->getMapPoint(s.first);
        if (lm) cull_if_weak(s.first, lm);
    }
    bstop_localba_ = false;                                            // optimizer.cpp:896: a stop request is consumed by the BA it interrupted
}

// ---------------------------------------------------------------------------------------------------------------
// 8f-4: Optimizer::looseBA (/root/reference/src/optimizer.cpp:900-1671) and Optimizer::fullBA (:1674-2331) - the same
// residual blocks and the same Ceres configuration as localBA over bigger windows (a loop's keyframes / the whole map),
// so the flattening above and the same solve kernel serve them.  What differs is the window rule, the iteration budget
// and the write-back, restated below.  Compile these two with -DOV2_EXTERNAL_LOOSE_FULL_BA on the reference side (an
// #ifndef around the two bodies, like localBA's); without the define the reference keeps its Ceres versions.
namespace {

// keyframes [first, last]: the first `nmincst` that exist are constant, the others are optimised and bring their 3-D
// keypoints' map points in (ascending map-point id: the reference collects them in a std::set)
void window_of_range(MapManager& map, Window& win, const int first, const int last, const bool stereo, std::vector<int>& lm_order) {
    const size_t nmincst = stereo ? 1 : 2;
    size_t ncst = 0;
    std::set<int> lmids;
    for (int kfid = first; kfid <= last; ++kfid) {
        auto kf = map.getKeyframe(kfid);
        if (!kf) continue;
        const bool constant = ncst < nmincst;
        if (constant) ncst++;
        win.add_camera(kfid, kf, constant);
        if (!constant)
            for (const auto& kp : kf->getKeypoints3d()) lmids.insert(kp.lmid_);
    }
    lm_order.assign(lmids.begin(), lmids.end());
}

// world point of landmark l from its anchor keyframe's CURRENT pose in the map (optimizer.cpp:1497-1511, :2262-2275)
bool world_point(const Window& win, size_t l, Eigen::Vector3d& out) {
    const double invd = win.lm_invdepth[l];
    if (1.0 / invd <= 0.0) return false;
    auto ait = win.cam_of_kf.find(win.lms[l]->kfid_);
    if (ait == win.cam_of_kf.end()) return false;
    auto kfa = win.kfs[ait->second];
    const auto kp = kfa->getKeypointById(win.lmids[l]);
    out = kfa->getTwc() * ((1.0 / invd) * kfa->pcalib_leftcam_->iK_ * Eigen::Vector3d(kp.unpx_.x, kp.unpx_.y, 1.0));
    return true;
}

void cull_bad(MapManager& map, const std::set<int>& bad, const int newest_kfid) {
    for (int lmid : bad) {
        auto lm = map.getMapPoint(lmid);
        if (!lm) continue;
        if (lm->isBad()) { map.removeMapPoint(lmid); continue; }
        if (lm->getKfObsSet().size() < 3 && lm->kfid_ < newest_kfid - 3 && !lm->isobs_) map.removeMapPoint(lmid);
    }
}

}  // namespace

#ifdef OV2_EXTERNAL_LOOSE_FULL_BA
void Optimizer::looseBA(const int inikfid, const int nkfid, const bool buse_robust_cost)
{
    auto pnew = pmap_->getKeyframe(nkfid);
    if (!pnew) return;
    Frame& newframe = *pnew;
    ov2_ctx* ctx = ba_context();
    if (!ctx) { std::cerr << "[ov2b200] looseBA: no CUDA device (no CPU fallback)\n"; return; }
    if (!pslamstate_->buse_inv_depth_) { std::cerr << "[ov2b200] looseBA: only the anchored inverse-depth parametrisation is built\n"; return; }
    const bool stereo = pslamstate_->stereo_;
    Window win;
    std::vector<int> lm_order;
    window_of_range(*pmap_, win, inikfid, nkfid, stereo, lm_order);          // optimizer.cpp:989-1020
    flatten_landmarks(*pmap_, win, lm_order, newframe.kfid_, stereo);        // :1023-1226
    fix_gauge_and_capacity(win, stereo, "looseBA");                          // :1228-1239
    if (win.obs_cam.empty()) return;
    double K[4], Kr[4] = {0, 0, 0, 0}, Trl[7] = {0, 0, 0, 0, 0, 0, 1};
    ov2_ba_problem pb;
    make_problem(win, win, newframe, stereo, K, Kr, Trl, pb);
    ov2_ba_opts op;
    op.max_iters_robust = 5; op.max_iters_refine = 0;                         // one solve: :1297-1310
    op.huber_th = pslamstate_->robust_mono_th_; op.function_tolerance = 1.e-4;
    op.use_robust = buse_robust_cost ? 1 : 0;
    op.apply_l2_after_robust = 0;                                             // no refinement solve in looseBA
    op.refine_loss = -1;
    ov2_ba_result res;
    std::vector<uint8_t> flags(win.obs_cam.size(), 0);
    const Sophus::SE3d iniTnewkfw = newframe.getTcw();                        // :1452
    if (ov2_localba_solve(ctx, &pb, &op, &res, flags.data()) != OV2_OK) {
        std::cerr << "[ov2b200] looseBA: " << ov2_last_error(ctx) << "\n";
        return;
    }
    // ---- write-back (:1322-1671)
    std::set<int> bad;
    for (size_t i = 0; i < flags.size(); ++i)
        if (flags[i] & 1) bad.insert(win.lmids[win.obs_lm[i]]);
    std::lock_guard<std::mutex> lock2(pmap_->optim_mutex_);
    std::lock_guard<std::mutex> lock(pmap_->map_mutex_);
    // the reference computes the landmarks' world points from the anchors' poses BEFORE the keyframes move (:1476-1521)
    std::vector<std::pair<int, Eigen::Vector3d>> wpts;
    for (size_t l = 0; l < win.lmids.size(); ++l) {
        if (win.lms[l]->isBad()) { bad.insert(win.lmids[l]); continue; }
        Eigen::Vector3d w;
        if (world_point(win, l, w)) wpts.emplace_back(win.lmids[l], w);
        else bad.insert(win.lmids[l]);
    }
    for (const auto& lw : wpts) pmap_->updateMapPoint(lw.first, lw.second);
    const auto cnew = win.cam_of_kf.find(newframe.kfid_);
    const double* pn = &win.pose[7 * cnew->second];
    const Sophus::SE3d optTwnewkf(Eigen::Quaterniond(pn[6], pn[3], pn[4], pn[5]), Eigen::Vector3d(pn[0], pn[1], pn[2]));
    for (size_t c = 0; c < win.kfids.size(); ++c) {
        if (win.pose_const[c]) continue;
        const double* p = &win.pose[7 * c];
        win.kfs[c]->setTwc(Sophus::SE3d(Eigen::Quaterniond(p[6], p[3], p[4], p[5]), Eigen::Vector3d(p[0], p[1], p[2])));
    }
    // keyframes created after the loop keyframe follow it rigidly, with the map points they anchor (:1541-1587)
    std::set<int> moved;
    const std::set<int> in_window(win.lmids.begin(), win.lmids.end());
    for (int kfid = newframe.kfid_ + 1; kfid <= pmap_->nkfid_; ++kfid) {
        if (win.cam_of_kf.count(kfid)) continue;
        auto kf = pmap_->getKeyframe(kfid);
        if (!kf) continue;
        const Sophus::SE3d updTwkf = optTwnewkf * (iniTnewkfw * kf->getTwc());
        for (const auto& kp : kf->getKeypoints3d()) {
            if (moved.count(kp.lmid_) || in_window.count(kp.lmid_)) continue;
            auto lm = pmap_->getMapPoint(kp.lmid_);
            if (!lm) { pmap_->removeMapPointObs(kp.lmid_, kfid); continue; }
            if (lm->kfid_ == kfid) {
                pmap_->updateMapPoint(kp.lmid_, updTwkf * kf->projWorldToCam(lm->getPoint()));
                moved.insert(lm->lmid_);
            }
        }
        kf->setTwc(updTwkf);
    }
    for (size_t i = 0; i < flags.size(); ++i) {                              // rejected right-camera observations (:1589-1600)
        if (!(flags[i] & 1) || win.obs_type[i] == 0) continue;
        win.kfs[win.obs_cam[i]]->removeStereoKeypointById(win.lmids[win.obs_lm[i]]);
    }
    for (size_t i = 0; i < flags.size(); ++i) {                              // rejected left-camera observations (:1602-1617)
        if (!(flags[i] & 1) || win.obs_type[i] != 0) continue;
        const int kfid = win.kfids[win.obs_cam[i]], lmid = win.lmids[win.obs_lm[i]];
        pmap_->removeMapPointObs(lmid, kfid);
        if (kfid == pmap_->pcurframe_->kfid_) pmap_->removeObsFromCurFrameById(lmid);
    }
    cull_bad(*pmap_, bad, newframe.kfid_);                                    // :1619-1647
    pmap_->pcurframe_->setTwc(optTwnewkf * (iniTnewkfw * pmap_->pcurframe_->getTwc()));   // :1649-1653
}

void Optimizer::fullBA(const bool buse_robust_cost)
{
    auto pfirst = pmap_->getKeyframe(0);
    if (!pfirst) return;
    Frame& newframe = *pfirst;                                                // calibration holder (:1676)
    ov2_ctx* ctx = ba_context();
    if (!ctx) { std::cerr << "[ov2b200] fullBA: no CUDA device (no CPU fallback)\n"; return; }
    if (!pslamstate_->buse_inv_depth_) { std::cerr << "[ov2b200] fullBA: only the anchored inverse-depth parametrisation is built\n"; return; }
    const bool stereo = pslamstate_->stereo_;
    Window win;
    std::vector<int> lm_order;
    window_of_range(*pmap_, win, 0, pmap_->nkfid_, stereo, lm_order);        // :1752-1790
    // fullBA has no `kfid > newframe.kfid_` filter worth the name: every keyframe of the map is in the window
    flatten_landmarks(*pmap_, win, lm_order, pmap_->nkfid_, stereo);         // :1794-1990
    fix_gauge_and_capacity(win, stereo, "fullBA");                           // :1992-2003
    if (win.obs_cam.empty()) return;
    double K[4], Kr[4] = {0, 0, 0, 0}, Trl[7] = {0, 0, 0, 0, 0, 0, 1};
    ov2_ba_problem pb;
    make_problem(win, win, newframe, stereo, K, Kr, Trl, pb);
    ov2_ba_opts op;
    op.max_iters_robust = 100; op.max_iters_refine = 100;                     // :2055-2061, :2149 (same options object)
    op.huber_th = pslamstate_->robust_mono_th_; op.function_tolerance = 1.e-6;   // Ceres' default: fullBA does not set it
    op.use_robust = buse_robust_cost ? 1 : 0;
    // the reference refines only when the first scan rejected something (:2140); the solve kernel refines whenever asked
    // to, which is the same thing unless nothing was rejected - and then the refinement starts at a converged point with
    // the same residual set and returns at its first iteration
    op.apply_l2_after_robust = pslamstate_->apply_l2_after_robust_ ? 1 : 0;
    op.refine_loss = -1;
    ov2_ba_result res;
    std::vector<uint8_t> flags(win.obs_cam.size(), 0);
    if (ov2_localba_solve(ctx, &pb, &op, &res, flags.data()) != OV2_OK) {
        std::cerr << "[ov2b200] fullBA: " << ov2_last_error(ctx) << "\n";
        return;
    }
    // ---- write-back (:2180-2331)
    std::set<int> bad;
    std::lock_guard<std::mutex> lock(pmap_->map_mutex_);
    for (size_t i = 0; i < flags.size(); ++i) {
        if (!flags[i]) continue;
        const int kfid = win.kfids[win.obs_cam[i]], lmid = win.lmids[win.obs_lm[i]];
        if (win.obs_type[i] == 0) {
            pmap_->removeMapPointObs(lmid, kfid);
            if (kfid == pmap_->pcurframe_->kfid_) pmap_->removeObsFromCurFrameById(lmid);
        } else {
            win.kfs[win.obs_cam[i]]->removeStereoKeypointById(lmid);
        }
        bad.insert(lmid);
    }
    for (size_t c = 0; c < win.kfids.size(); ++c) {
        if (win.pose_const[c]) continue;
        const double* p = &win.pose[7 * c];
        win.kfs[c]->setTwc(Sophus::SE3d(Eigen::Quaterniond(p[6], p[3], p[4], p[5]), Eigen::Vector3d(p[0], p[1], p[2])));
    }
    for (size_t l = 0; l < win.lmids.size(); ++l) {
        const int lmid = win.lmids[l];
        if (win.lms[l]->isBad()) { pmap_->removeMapPoint(lmid); bad.erase(lmid); continue; }
        Eigen::Vector3d w;
        if (!world_point(win, l, w)) { pmap_->removeMapPoint(lmid); bad.erase(lmid); continue; }
        pmap_->updateMapPoint(lmid, w, win.lm_invdepth[l]);
    }
    cull_bad(*pmap_, bad, pmap_->nkfid_);
}
#endif  // OV2_EXTERNAL_LOOSE_FULL_BA

