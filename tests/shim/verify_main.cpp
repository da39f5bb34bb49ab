// Drives both drop-in files the way cpp_code/test/sfm.cpp:140-166 drives the reference, with the batch hooks:
//   esfm_prepare_all_pairs -> (per-call answers) -> esfm_verify_all_pairs -> the loop over estimate2D2D_E5P_RANSAC again (lookups), and once
//   more with every pair's last match dropped (no longer the batch's matches: computed per call).
// usage: verify_main <in file> <out file>
//   in : int32 n_frames; per frame: double K[9]; int32 n_kp; float kp[n_kp][2]; uint8 desc[n_kp][32]
//   out: per pair with more than 20 matches, loop order: int32 i, j, n_matches, lookup equals per call, altered equals its per-call answer
#include <cstdio>
#include <cstring>
#include <vector>

#include "estimate_motion.h"

namespace p3dv {
bool esfm_verify_all_pairs(std::vector<frame_t>& frames, double ransac_thre, double ransac_prob, int num_min_pair);
}

namespace {
struct Answer {
    bool ok = false;
    std::vector<cv::DMatch> inliers;
    Eigen::Matrix4f T;
};

bool same(const Answer& a, const Answer& b) {
    return a.ok == b.ok && a.inliers.size() == b.inliers.size() &&
           (a.inliers.empty() || std::memcmp(a.inliers.data(), b.inliers.data(), a.inliers.size() * sizeof(cv::DMatch)) == 0) &&
           std::memcmp(&a.T, &b.T, sizeof a.T) == 0;
}
}  // namespace

int main(int argc, char** argv) {
    if (argc < 3) return 2;
    FILE* f = std::fopen(argv[1], "rb");
    if (!f) return 3;
    int n = 0;
    if (std::fread(&n, 4, 1, f) != 1) return 4;
    std::vector<p3dv::frame_t> frames((size_t)n);
    std::vector<std::vector<unsigned char> > desc((size_t)n);
    for (int i = 0; i < n; ++i) {
        p3dv::frame_t& fr = frames[(size_t)i];
        fr.frame_id = (unsigned)i;            // sfm.cpp numbers the frames by position
        double K[9];
        int nk = 0;
        if (std::fread(K, 8, 9, f) != 9 || std::fread(&nk, 4, 1, f) != 1) return 4;
        for (int r = 0; r < 3; ++r)
            for (int c = 0; c < 3; ++c) fr.K_cam(r, c) = (float)K[3 * r + c];
        fr.keypoints.resize((size_t)nk);
        for (int k = 0; k < nk; ++k) if (std::fread(&fr.keypoints[(size_t)k].pt, 4, 2, f) != 2) return 4;
        desc[(size_t)i].resize((size_t)nk * 32 + 1);
        if (nk && std::fread(desc[(size_t)i].data(), 32, (size_t)nk, f) != (size_t)nk) return 4;
        fr.descriptors.flags_type = CV_8UC1;
        fr.descriptors.rows = nk;
        fr.descriptors.cols = 32;
        fr.descriptors.data = desc[(size_t)i].data();
        fr.descriptors.step.v = 32;
    }
    std::fclose(f);
    const int num_min_pair = 20;
    if (!p3dv::esfm_prepare_all_pairs(frames, 'O', 0.8, false)) return 5;
    p3dv::FeatureMatching fm;
    p3dv::MotionEstimator ee;
    std::vector<std::vector<cv::DMatch> > matches;
    std::vector<Answer> per_call, altered_per_call;
    for (int i = 0; i < n; ++i)
        for (int j = 0; j < i; ++j) {
            std::vector<cv::DMatch> m;
            if (!fm.matchFeaturesORB(frames[(size_t)i], frames[(size_t)j], m)) return 6;
            matches.push_back(m);
            Answer a, b;
            if (m.size() > (size_t)num_min_pair) {
                a.ok = ee.estimate2D2D_E5P_RANSAC(frames[(size_t)i], frames[(size_t)j], m, a.inliers, a.T);
                std::vector<cv::DMatch> shorter(m.begin(), m.end() - 1);
                b.ok = ee.estimate2D2D_E5P_RANSAC(frames[(size_t)i], frames[(size_t)j], shorter, b.inliers, b.T);
            }
            per_call.push_back(a);
            altered_per_call.push_back(b);
        }
    if (!p3dv::esfm_verify_all_pairs(frames, 1.0, 0.99, num_min_pair)) return 7;
    FILE* o = std::fopen(argv[2], "wb");
    if (!o) return 3;
    size_t k = 0;
    for (int i = 0; i < n; ++i)
        for (int j = 0; j < i; ++j, ++k) {
            std::vector<cv::DMatch>& m = matches[k];
            if (m.size() <= (size_t)num_min_pair) continue;
            Answer a, b;
            a.ok = ee.estimate2D2D_E5P_RANSAC(frames[(size_t)i], frames[(size_t)j], m, a.inliers, a.T);
            std::vector<cv::DMatch> shorter(m.begin(), m.end() - 1);
            b.ok = ee.estimate2D2D_E5P_RANSAC(frames[(size_t)i], frames[(size_t)j], shorter, b.inliers, b.T);
            const int rec[5] = {i, j, (int)m.size(), same(a, per_call[k]) ? 1 : 0, same(b, altered_per_call[k]) ? 1 : 0};
            std::fwrite(rec, 4, 5, o);
        }
    std::fclose(o);
    return 0;
}
