// estimate_motion_gpu.cpp -- drop-in for the two-view part of EasySFM's cpp_code/src/estimate_motion.cpp (SURVEY 8f rank 1).
//
// Keeps the two public methods of p3dv::MotionEstimator that the all-pairs loop calls (cpp_code/test/sfm.cpp:165-166) with their
// reference signatures and defaults (cpp_code/include/estimate_motion.h:17-20, :26-27):
//     estimate2D2D_E5P_RANSAC   estimate_motion.cpp:27-97    cv::findEssentialMat(RANSAC) -> inlier matches -> cv::recoverPose -> T
//     getDepthFast              estimate_motion.cpp:234-283  cv::triangulatePoints of every random_rate-th match -> mean point norm
// and forwards them to the C ABI (esfm_two_view_batch / esfm_two_view_depth, include/esfm_match.h).  Build: compile this file instead of the
// two functions in estimate_motion.cpp (wrap them in #ifndef ESFM_GPU) and link libesfm_match.so, as for feature_matching_gpu.cpp
// (INTEGRATION.md).  The other methods of the class (PnP, triangulation, outlier filter) stay in estimate_motion.cpp.
// No CPU fallback: without a B200 the calls fail and return false.  `show` (GUI windows) is not carried across the C ABI.
// After p3dv::esfm_verify_all_pairs (feature_matching_gpu.cpp) a call whose matches are the verified batch's matches of (frame_1, frame_2),
// with the hook's ransac_thre / ransac_prob, is a lookup: the batch keyed the pair's sampler exactly as this file does, so both answers are
// the same bytes.  Any other call is computed as before.
#include <chrono>
#include <cstdlib>
#include <cstring>
#include <iostream>
#include <vector>

#include "estimate_motion.h"
#include "esfm_match.h"
#include "esfm_verified.h"

namespace p3dv {

namespace {

struct MotionState {
    esfm_ctx_t* ctx = nullptr;
    ~MotionState() {
        if (ctx) esfm_destroy(ctx);
    }
};

esfm_ctx_t* motion_ctx() {
    static MotionState s;
    if (!s.ctx) {
        const char* dev = std::getenv("ESFM_DEVICE");
        if (esfm_init(dev ? std::atoi(dev) : 0, nullptr, &s.ctx) != ESFM_OK) {
            std::cerr << "esfm_init failed: " << esfm_last_error() << std::endl;
            s.ctx = nullptr;
        }
    }
    return s.ctx;
}

// pts1[k] = frame_1.keypoints[matches[k].queryIdx].pt, pts2[k] = frame_2.keypoints[matches[k].trainIdx].pt (estimate_motion.cpp:36-40)
void gather(const frame_t& f1, const frame_t& f2, const std::vector<cv::DMatch>& matches, std::vector<float>& p1, std::vector<float>& p2) {
    p1.resize(2 * matches.size());
    p2.resize(2 * matches.size());
    for (size_t i = 0; i < matches.size(); ++i) {
        const cv::Point2f a = f1.keypoints[matches[i].queryIdx].pt, b = f2.keypoints[matches[i].trainIdx].pt;
        p1[2 * i] = a.x; p1[2 * i + 1] = a.y;
        p2[2 * i] = b.x; p2[2 * i + 1] = b.y;
    }
}

void camera(const frame_t& f, double (&K)[9]) {
    for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 3; ++c) K[3 * r + c] = (double)f.K_cam(r, c);     // cv::eigen2cv(cur_frame_1.K_cam, camera_mat), :43
}

void pose_to_T(const esfm_two_view_t& tv, Eigen::Matrix4f& T) {
    for (int r = 0; r < 3; ++r) {
        for (int c = 0; c < 3; ++c) T(r, c) = (float)tv.R[3 * r + c];         // T.block(0, 0, 3, 3) = R, :76
        T(r, 3) = (float)tv.t[r];                                              // T.block(0, 3, 3, 1) = t, :77
        T(3, r) = 0.f;
    }
    T(3, 3) = 1.f;
}

// The verified batch's answer for this call, if it has one: same pair, same match records (count and bytes), same parameters.
bool lookup(const frame_t& f1, const frame_t& f2, const std::vector<cv::DMatch>& matches, double ransac_thre, double ransac_prob,
            std::vector<cv::DMatch>& inlier_matches, Eigen::Matrix4f& T) {
    const esfm_shim::VerifiedBatch& v = esfm_shim::verified();
    if (!v.inliers || ransac_thre != v.ransac_thre || ransac_prob != v.ransac_prob || (int64_t)matches.size() <= (int64_t)v.min_pair) return false;
    auto it = v.index.find(((uint64_t)f1.frame_id << 32) | (uint64_t)f2.frame_id);
    if (it == v.index.end()) return false;
    const esfm_dmatch_t* m = nullptr;
    int n = 0;
    if (esfm_results_pair_at(v.matches, it->second, nullptr, nullptr, &m, &n) != ESFM_OK || (size_t)n != matches.size()) return false;
    if (n && std::memcmp(m, matches.data(), (size_t)n * sizeof(esfm_dmatch_t)) != 0) return false;
    const esfm_dmatch_t* inl = nullptr;
    int ni = 0;
    if (esfm_results_pair_at(v.inliers, it->second, nullptr, nullptr, &inl, &ni) != ESFM_OK) return false;
    const size_t before = inlier_matches.size();
    inlier_matches.resize(before + (size_t)ni);                                 // appended, as the reference does (:54-60)
    if (ni) std::memcpy(static_cast<void*>(&inlier_matches[before]), inl, (size_t)ni * sizeof(esfm_dmatch_t));
    pose_to_T(v.tv[(size_t)it->second], T);
    return true;
}

}  // namespace

bool MotionEstimator::estimate2D2D_E5P_RANSAC(frame_t& cur_frame_1, frame_t& cur_frame_2, std::vector<cv::DMatch>& matches,
                                              std::vector<cv::DMatch>& inlier_matches, Eigen::Matrix4f& T, double ransac_thre, double ransac_prob, bool show) {
    (void)show;
    std::chrono::steady_clock::time_point tic = std::chrono::steady_clock::now();
    if (lookup(cur_frame_1, cur_frame_2, matches, ransac_thre, ransac_prob, inlier_matches, T)) {
        std::chrono::duration<double> time_used = std::chrono::duration_cast<std::chrono::duration<double>>(std::chrono::steady_clock::now() - tic);
        std::cout << "Estimate Motion [2D-2D] (verified batch) cost = " << time_used.count() << " seconds. " << std::endl;
        std::cout << "Find [" << inlier_matches.size() << "] inlier matches from [" << matches.size() << "] total matches." << std::endl;
        return true;
    }
    esfm_ctx_t* ctx = motion_ctx();
    if (!ctx) return false;
    std::vector<float> p1, p2;
    gather(cur_frame_1, cur_frame_2, matches, p1, p2);
    double K[9];
    camera(cur_frame_1, K);
    esfm_two_view_params_t prm;
    esfm_two_view_default_params(&prm);
    prm.ransac_thre = ransac_thre;
    prm.ransac_prob = ransac_prob;
    prm.seed = esfm_shim::ransac_seed();
    // the sampler key of this pair: its two frame ids, so a pair draws the same hypotheses however the loop reaches it
    prm.first_pair = ((uint64_t)cur_frame_1.frame_id << 32) | (uint64_t)cur_frame_2.frame_id;
    const int64_t off[2] = {0, (int64_t)matches.size()};
    std::vector<unsigned char> mask(matches.size() + 1);
    esfm_two_view_t tv;
    if (esfm_two_view_batch(ctx, 1, off, p1.data(), p2.data(), K, 0, &prm, mask.data(), &tv) != ESFM_OK) {
        std::cerr << "esfm_two_view_batch failed: " << esfm_last_error() << std::endl;
        return false;
    }
    for (size_t i = 0; i < matches.size(); ++i)
        if (mask[i]) inlier_matches.push_back(matches[i]);                    // appended, as the reference does (:54-60)
    pose_to_T(tv, T);
    std::chrono::duration<double> time_used = std::chrono::duration_cast<std::chrono::duration<double>>(std::chrono::steady_clock::now() - tic);
    std::cout << "Estimate Motion [2D-2D] cost = " << time_used.count() << " seconds. " << std::endl;
    std::cout << "Find [" << inlier_matches.size() << "] inlier matches from [" << matches.size() << "] total matches." << std::endl;
    return true;      // (the reference returns 1 unconditionally; a pair without a model leaves inlier_matches empty and T = [0 | 0])
}

bool MotionEstimator::getDepthFast(frame_t& cur_frame_1, frame_t& cur_frame_2, Eigen::Matrix4f& T_21, const std::vector<cv::DMatch>& matches,
                                   double& appro_depth, int random_rate) {
    esfm_ctx_t* ctx = motion_ctx();
    if (!ctx) return false;
    std::vector<float> p1, p2;
    gather(cur_frame_1, cur_frame_2, matches, p1, p2);
    double K[9], R[9], t[3];
    camera(cur_frame_1, K);
    for (int r = 0; r < 3; ++r) {
        for (int c = 0; c < 3; ++c) R[3 * r + c] = (double)T_21(r, c);
        t[r] = (double)T_21(r, 3);
    }
    int32_t used = 0;
    if (esfm_two_view_depth(ctx, (int64_t)matches.size(), p1.data(), p2.data(), K, R, t, random_rate, &appro_depth, &used) != ESFM_OK) {
        std::cerr << "esfm_two_view_depth failed: " << esfm_last_error() << std::endl;
        return false;
    }
    std::cout << "Mean relative depth is about " << appro_depth << " * baseline length. " << std::endl;
    return true;
}

}  // namespace p3dv
