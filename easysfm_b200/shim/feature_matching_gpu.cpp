// feature_matching_gpu.cpp -- drop-in replacement for the two matching methods of p3dv::FeatureMatching
// (EasySFM cpp_code/src/feature_matching.cpp:71-158) and for detectFeaturesORB (:14-41), forwarding to libesfm_match.so through the C ABI.
//
// Build it INSTEAD of the two method bodies in feature_matching.cpp (see INTEGRATION.md): the signatures
// below are verbatim from cpp_code/include/feature_matching.h:17-21, so cpp_code/test/sfm.cpp compiles and
// runs unchanged -- initial-pair selection, 5-point RANSAC, PnP and Ceres BA consume the GPU matches.
//
//   * per-call path (unmodified caller, sfm.cpp:153,156): the two frames' descriptors are uploaded and matched
//     on the GPU for every call (esfm_match_descriptors).
//   * all-pairs path: call p3dv::esfm_prepare_all_pairs(frames, 'S'|'O', ratio, cross_check) once before the
//     pair loop (a one-line hook at sfm.cpp:131); every later matchFeatures* call on those frames with the same
//     ratio is a lookup into the precomputed result (esfm_results_pair).  ESFM_GPUS=N (N > 1) runs that pass on N GPUs
//     of the box from this one process (esfm_multi_*: ncclBroadcast of the bank, pairs dealt by work, matches merged).
//   * resume: p3dv::esfm_save_matches(path) after the prepare step writes the whole batch to a match file;
//     p3dv::esfm_load_matches(frames, 'S'|'O', ratio, path) in a later run makes the same lookups work without
//     matching again (and without touching the GPU).
//   * verification: p3dv::esfm_verify_all_pairs(frames, ransac_thre, ransac_prob, num_min_pair) after the prepare (or load) step
//     verifies every pair of the batch on the device (esfm_two_view_results; ESFM_GPUS=N > 1: on N GPUs); later
//     MotionEstimator::estimate2D2D_E5P_RANSAC calls with a pair's unaltered matches are lookups (estimate_motion_gpu.cpp).
//
// Semantics kept from the reference: matches are APPENDED (push_back, :90/:135), ascending queryIdx, imgIdx = 0,
// returns true; ratio test in double (:88/:133); the stdout summary lines (:81,96-97 / :126,141-142).
// Differences, deliberate (SURVEY.md F2/F3): matchFeaturesSURF is an EXACT L2 brute-force search (the reference
// calls the approximate cv::FlannBasedMatcher, :120); `show` is accepted and ignored (GUI only, :99-110);
// the mutual cross-check is off unless ESFM_CROSS_CHECK=1 or esfm_prepare_all_pairs(..., cross_check = true).
//
// This file needs the EasySFM headers (utility.h -> OpenCV, Eigen, PCL); for the compile check in this
// repository tests/shim/ provides a minimal stand-in for those headers.
#include <chrono>
#include <cstdlib>
#include <cstring>
#include <iostream>
#include <map>
#include <vector>

#include "feature_matching.h"  // EasySFM's own header: class p3dv::FeatureMatching, frame_t
#include "esfm_match.h"
#include "esfm_verified.h"

namespace p3dv {
namespace {

struct GpuState {
    esfm_ctx_t* ctx = nullptr;
    esfm_bank_t* bank = nullptr;          // all-pairs bank (esfm_prepare_all_pairs), one GPU
    esfm_multi_t* multi = nullptr;        // ... or several GPUs (ESFM_GPUS > 1)
    esfm_multi_bank_t* mbank = nullptr;
    esfm_results_t* results = nullptr;
    esfm_kind kind = ESFM_KIND_F32X64;
    double ratio = 0.0;
    bool cross_check = false;             // the mode of the prepared / loaded batch; also what the per-call path uses from then on
    bool have_mode = false;
    std::map<unsigned int, int> frame_index;  // frame_t::frame_id -> bank slot
    ~GpuState() {
        if (results) esfm_results_destroy(results);
        if (mbank) esfm_multi_bank_destroy(mbank);
        if (multi) esfm_multi_destroy(multi);
        if (bank) esfm_bank_destroy(bank);
        if (ctx) esfm_destroy(ctx);
    }
};

GpuState& state() {
    static GpuState s;
    return s;
}

bool env_cross_check() {
    const char* e = std::getenv("ESFM_CROSS_CHECK");
    return e && e[0] == '1';
}

// One cross-check mode per process: $ESFM_CROSS_CHECK until a batch is prepared or loaded, that batch's mode afterwards --
// so a lookup and a per-call fallback of the same run can never disagree.
bool effective_cross_check();

int env_gpus() {
    const char* e = std::getenv("ESFM_GPUS");
    const int n = e ? std::atoi(e) : 1;
    return n < 1 ? 1 : n;
}

bool ensure_ctx() {
    GpuState& s = state();
    if (s.ctx) return true;
    const char* dev = std::getenv("ESFM_DEVICE");
    if (esfm_init(dev ? std::atoi(dev) : 0, nullptr, &s.ctx) != ESFM_OK) {
        std::cerr << "esfm_init failed: " << esfm_last_error() << std::endl;  // no CPU fallback: report and fail
        return false;
    }
    return true;
}

bool effective_cross_check() {
    GpuState& s = state();
    return s.have_mode ? s.cross_check : env_cross_check();
}

bool check_mat(const cv::Mat& m, esfm_kind kind) {
    if (m.rows == 0) return true;
    if (kind == ESFM_KIND_F32X64) return m.type() == CV_32FC1 && m.cols == 64;
    return m.type() == CV_8UC1 && m.cols == 32;
}

bool match_common(esfm_kind kind, const char* tag, frame_t& f1, frame_t& f2, std::vector<cv::DMatch>& matches, double ratio) {
    static_assert(sizeof(cv::DMatch) == sizeof(esfm_dmatch_t), "esfm_dmatch_t must be layout-identical to cv::DMatch");
    GpuState& s = state();
    std::chrono::steady_clock::time_point tic = std::chrono::steady_clock::now();
    const cv::Mat& q = f1.descriptors;  // cur_frame_1 is the query side (knnMatch(cur_frame_1, cur_frame_2), :80/:125)
    const cv::Mat& t = f2.descriptors;
    if (!check_mat(q, kind) || !check_mat(t, kind)) {
        std::cerr << "match" << tag << ": descriptors must be " << (kind == ESFM_KIND_F32X64 ? "CV_32FC1 x 64" : "CV_8UC1 x 32") << std::endl;
        return false;
    }
    const size_t before = matches.size();
    bool done = false;
    if (s.results && s.kind == kind && s.ratio == ratio && s.cross_check == effective_cross_check()) {  // all-pairs lookup
        auto a = s.frame_index.find(f1.frame_id), b = s.frame_index.find(f2.frame_id);
        if (a != s.frame_index.end() && b != s.frame_index.end()) {
            const esfm_dmatch_t* p = nullptr;
            int n = 0;
            if (esfm_results_pair(s.results, a->second, b->second, &p, &n) == ESFM_OK) {
                matches.resize(before + (size_t)n);
                if (n) std::memcpy(static_cast<void*>(&matches[before]), p, (size_t)n * sizeof(esfm_dmatch_t));
                done = true;
            }
        }
    }
    if (!done) {  // per-call path
        if (!ensure_ctx()) return false;
        std::vector<esfm_dmatch_t> buf((size_t)std::max(q.rows, 1));
        int n = 0;
        const int rc = esfm_match_descriptors(s.ctx, kind, q.data, q.rows, (size_t)q.step, t.data, t.rows, (size_t)t.step,
                                              kind == ESFM_KIND_F32X64 ? 64 : 32, ratio, effective_cross_check() ? 1 : 0,
                                              buf.data(), (int)buf.size(), &n);
        if (rc != ESFM_OK) {
            std::cerr << "match" << tag << " failed: " << esfm_last_error() << std::endl;
            return false;
        }
        matches.resize(before + (size_t)n);
        if (n) std::memcpy(static_cast<void*>(&matches[before]), buf.data(), (size_t)n * sizeof(esfm_dmatch_t));
    }
    std::cout << "Initial matching done." << std::endl;
    std::chrono::steady_clock::time_point toc = std::chrono::steady_clock::now();
    std::chrono::duration<double> time_used = std::chrono::duration_cast<std::chrono::duration<double>>(toc - tic);
    std::cout << "match " << tag << " cost = " << time_used.count() << " seconds. " << std::endl;
    std::cout << "# Correspondence: Initial [ " << q.rows << " ]  Filtered by Lowe ratio test [ " << matches.size() << " ]" << std::endl;
    return true;
}

}  // namespace

// One device pass over all N(N-1)/2 pairs in the reference's loop order (sfm.cpp:140-161: query = frames[i],
// train = frames[j], j < i).  feature = 'S' (SURF, L2) or 'O' (ORB, Hamming) as in sfm.cpp:52.
bool esfm_prepare_all_pairs(std::vector<frame_t>& frames, char feature, double ratio_thre, bool cross_check) {
    GpuState& s = state();
    const int gpus = env_gpus();
    esfm_shim::verified().clear();
    if (s.results) { esfm_results_destroy(s.results); s.results = nullptr; }
    if (s.mbank) { esfm_multi_bank_destroy(s.mbank); s.mbank = nullptr; }
    if (s.bank) { esfm_bank_destroy(s.bank); s.bank = nullptr; }
    s.frame_index.clear();
    s.kind = feature == 'O' ? ESFM_KIND_B256 : ESFM_KIND_F32X64;
    s.ratio = ratio_thre;
    s.cross_check = cross_check;
    s.have_mode = true;
    int rc = ESFM_OK;
    if (gpus > 1) {
        if (!s.multi) rc = esfm_multi_init(gpus, nullptr, &s.multi);
        if (rc == ESFM_OK) rc = esfm_multi_bank_create(s.multi, s.kind, (int)frames.size(), &s.mbank);
    } else {
        if (!ensure_ctx()) return false;
        rc = esfm_bank_create(s.ctx, s.kind, (int)frames.size(), &s.bank);
    }
    for (size_t i = 0; rc == ESFM_OK && i < frames.size(); ++i) {
        const cv::Mat& d = frames[i].descriptors;
        if (!check_mat(d, s.kind)) { std::cerr << "esfm_prepare_all_pairs: frame " << i << " has the wrong descriptor type" << std::endl; return false; }
        const int cols = d.rows ? d.cols : (s.kind == ESFM_KIND_F32X64 ? 64 : 32);
        rc = gpus > 1 ? esfm_multi_bank_set_frame(s.mbank, (int)i, d.data, d.rows, cols, (size_t)d.step)
                      : esfm_bank_set_frame(s.bank, (int)i, d.data, d.rows, cols, (size_t)d.step);
        s.frame_index[frames[i].frame_id] = (int)i;
    }
    if (rc == ESFM_OK) rc = gpus > 1 ? esfm_multi_bank_commit(s.mbank) : esfm_bank_commit(s.bank);
    if (rc == ESFM_OK)
        rc = gpus > 1 ? esfm_multi_match_all_pairs(s.mbank, ratio_thre, cross_check ? 1 : 0, ESFM_KEEP_MATCHES, &s.results)
                      : esfm_match_all_pairs(s.bank, ratio_thre, cross_check ? 1 : 0, &s.results);
    if (rc != ESFM_OK) {
        std::cerr << "esfm_prepare_all_pairs failed: " << esfm_last_error() << std::endl;
        return false;
    }
    return true;
}

// Persist the batch computed by esfm_prepare_all_pairs (SURVEY 8f: the reference keeps matches in RAM only, sfm.cpp:130-197).
bool esfm_save_matches(const char* path) {
    GpuState& s = state();
    if (!s.results) { std::cerr << "esfm_save_matches: nothing prepared" << std::endl; return false; }
    if (esfm_results_save(s.results, path) != ESFM_OK) { std::cerr << "esfm_save_matches failed: " << esfm_last_error() << std::endl; return false; }
    return true;
}

// Resume: load a match file written for the same frame list (same order), feature kind and ratio.  No device is needed;
// every later matchFeatures* call on those frames with that ratio is a lookup.
bool esfm_load_matches(std::vector<frame_t>& frames, char feature, double ratio_thre, const char* path) {
    GpuState& s = state();
    esfm_results_t* r = nullptr;
    if (esfm_results_load(path, &r) != ESFM_OK) { std::cerr << "esfm_load_matches failed: " << esfm_last_error() << std::endl; return false; }
    int kind = -1, cc = 0;
    double ratio = 0.0;
    esfm_results_params(r, &kind, &ratio, &cc);
    const esfm_kind want = feature == 'O' ? ESFM_KIND_B256 : ESFM_KIND_F32X64;
    if (kind != (int)want || ratio != ratio_thre) {
        std::cerr << "esfm_load_matches: " << path << " was matched with kind " << kind << ", ratio " << ratio << std::endl;
        esfm_results_destroy(r);
        return false;
    }
    // the file must belong to THIS frame list: stored row counts (version-2 files), pair ids and every match index are checked,
    // so a file saved for another image set cannot hand out-of-range indices to the RANSAC / triangulation code
    std::vector<int32_t> rows(frames.size());
    for (size_t i = 0; i < frames.size(); ++i) rows[i] = frames[i].descriptors.rows;
    if (esfm_results_validate(r, (int)rows.size(), rows.data()) != ESFM_OK) {
        std::cerr << "esfm_load_matches: " << path << " does not fit these frames: " << esfm_last_error() << std::endl;
        esfm_results_destroy(r);
        return false;
    }
    esfm_shim::verified().clear();
    if (s.results) esfm_results_destroy(s.results);
    s.results = r;
    s.kind = want;
    s.ratio = ratio_thre;
    s.cross_check = cc != 0;
    s.have_mode = true;
    s.frame_index.clear();
    for (size_t i = 0; i < frames.size(); ++i) s.frame_index[frames[i].frame_id] = (int)i;
    return true;
}

// The two-view step of the reference's loop (sfm.cpp:163-166: estimate2D2D_E5P_RANSAC on every pair with more than num_min_pair matches) for
// the whole prepared or loaded batch at once, on the device.  A frame's key points are frame_t::keypoints, its camera frame_t::K_cam (a pair
// uses its query frame's, as estimate_motion.cpp:43 does).  Frame ids must be the frames' positions, as the reference numbers them: the
// per-call path keys each pair's RANSAC samples by its frame ids, the batch by its positions, and the lookups rely on the two being equal.
bool esfm_verify_all_pairs(std::vector<frame_t>& frames, double ransac_thre, double ransac_prob, int num_min_pair) {
    GpuState& s = state();
    esfm_shim::VerifiedBatch& v = esfm_shim::verified();
    v.clear();
    if (!s.results) { std::cerr << "esfm_verify_all_pairs: call esfm_prepare_all_pairs or esfm_load_matches first" << std::endl; return false; }
    const int n = (int)frames.size();
    std::vector<int64_t> kp_off((size_t)n + 1, 0);
    for (int i = 0; i < n; ++i) {
        if (frames[(size_t)i].frame_id != (unsigned)i) {
            std::cerr << "esfm_verify_all_pairs: frame " << i << " has frame_id " << frames[(size_t)i].frame_id << " (ids must be 0..n-1)" << std::endl;
            return false;
        }
        kp_off[(size_t)i + 1] = kp_off[(size_t)i] + (int64_t)frames[(size_t)i].keypoints.size();
    }
    std::vector<float> xy((size_t)kp_off[(size_t)n] * 2 + 2);
    std::vector<double> K((size_t)n * 9 + 9);
    for (int i = 0; i < n; ++i) {
        const frame_t& f = frames[(size_t)i];
        for (size_t k = 0; k < f.keypoints.size(); ++k) {
            xy[2 * ((size_t)kp_off[(size_t)i] + k)] = f.keypoints[k].pt.x;
            xy[2 * ((size_t)kp_off[(size_t)i] + k) + 1] = f.keypoints[k].pt.y;
        }
        for (int r = 0; r < 3; ++r)
            for (int c = 0; c < 3; ++c) K[(size_t)i * 9 + 3 * r + c] = (double)f.K_cam(r, c);
    }
    esfm_two_view_params_t prm;
    esfm_two_view_default_params(&prm);
    prm.ransac_thre = ransac_thre;
    prm.ransac_prob = ransac_prob;
    prm.seed = esfm_shim::ransac_seed();
    int64_t n_pairs = 0;
    esfm_results_counts(s.results, &n_pairs, nullptr);
    v.tv.resize((size_t)std::max<int64_t>(n_pairs, 1));
    const int gpus = env_gpus();
    int rc = ESFM_OK;
    if (gpus > 1) {
        if (!s.multi) rc = esfm_multi_init(gpus, nullptr, &s.multi);
        if (rc == ESFM_OK)
            rc = esfm_multi_two_view_results(s.multi, s.results, n, kp_off.data(), xy.data(), K.data(), 1, &prm, num_min_pair, &v.inliers, v.tv.data());
    } else {
        if (!ensure_ctx()) return false;
        rc = esfm_two_view_results(s.ctx, s.results, n, kp_off.data(), xy.data(), K.data(), 1, &prm, num_min_pair, &v.inliers, v.tv.data());
    }
    if (rc != ESFM_OK) {
        std::cerr << "esfm_verify_all_pairs failed: " << esfm_last_error() << std::endl;
        v.clear();
        return false;
    }
    v.matches = s.results;
    v.ransac_thre = ransac_thre;
    v.ransac_prob = ransac_prob;
    v.min_pair = num_min_pair;
    for (int64_t k = 0; k < n_pairs; ++k) {
        int q = 0, t = 0;
        esfm_results_pair_at(s.results, k, &q, &t, nullptr, nullptr);
        v.index.emplace(((uint64_t)(uint32_t)q << 32) | (uint32_t)t, k);
    }
    return true;
}

// cpp_code/src/feature_matching.cpp:14-41 (decl feature_matching.h:13): cv::ORB::create(max_num)->detect + ->compute on cur_frame.rgb_image,
// filling cur_frame.keypoints and cur_frame.descriptors.  The device computes what cv2 4.13 computes, bit for bit and in the same order
// (esfm_orb_extract); `show` only opens a GUI window in the reference (:32-38) and is ignored.
bool FeatureMatching::detectFeaturesORB(frame_t& cur_frame, int max_num, bool show) {
    (void)show;
    if (!ensure_ctx()) return false;
    const cv::Mat& img = cur_frame.rgb_image;
    if (img.empty() || (img.type() != CV_8UC3 && img.type() != CV_8UC1)) {
        std::cerr << "detectFeaturesORB: rgb_image must be a non-empty CV_8UC3 or CV_8UC1 image" << std::endl;
        return false;
    }
    std::chrono::steady_clock::time_point tic = std::chrono::steady_clock::now();
    std::vector<esfm_keypoint_t> kp((size_t)(max_num > 0 ? max_num : 0) + 256);
    std::vector<unsigned char> desc(kp.size() * 32);
    int n = 0;
    int rc = esfm_orb_extract(state().ctx, img.data, img.rows, img.cols, img.channels(), (size_t)img.step, max_num, kp.data(), desc.data(),
                              (int)kp.size(), &n);
    if (rc == ESFM_ERR_CAPACITY && n > (int)kp.size()) {   // more Harris ties at the cut than the slack: once more with room for all
        kp.resize((size_t)n);
        desc.resize((size_t)n * 32);
        rc = esfm_orb_extract(state().ctx, img.data, img.rows, img.cols, img.channels(), (size_t)img.step, max_num, kp.data(), desc.data(), n, &n);
    }
    if (rc != ESFM_OK) {
        std::cerr << "esfm_orb_extract failed: " << esfm_last_error() << std::endl;
        return false;
    }
    cur_frame.keypoints.resize((size_t)n);
    for (int i = 0; i < n; ++i) {
        cv::KeyPoint& k = cur_frame.keypoints[(size_t)i];
        k.pt.x = kp[(size_t)i].x;
        k.pt.y = kp[(size_t)i].y;
        k.size = kp[(size_t)i].size;
        k.angle = kp[(size_t)i].angle;
        k.response = kp[(size_t)i].response;
        k.octave = kp[(size_t)i].octave;
        k.class_id = -1;
    }
    cur_frame.descriptors.create(n, 32, CV_8UC1);
    if (n) std::memcpy(cur_frame.descriptors.data, desc.data(), (size_t)n * 32);
    std::chrono::steady_clock::time_point toc = std::chrono::steady_clock::now();
    std::chrono::duration<double> time_used = std::chrono::duration_cast<std::chrono::duration<double>>(toc - tic);
    std::cout << "extract ORB cost = " << time_used.count() << " seconds. " << std::endl;    // :28-30
    std::cout << "Found [32 x " << n << "] features" << std::endl;
    return true;
}

bool FeatureMatching::matchFeaturesORB(frame_t& cur_frame_1, frame_t& cur_frame_2, std::vector<cv::DMatch>& matches,
                                       double ratio_thre, bool show) {
    (void)show;
    return match_common(ESFM_KIND_B256, "ORB", cur_frame_1, cur_frame_2, matches, ratio_thre);
}

bool FeatureMatching::matchFeaturesSURF(frame_t& cur_frame_1, frame_t& cur_frame_2, std::vector<cv::DMatch>& matches,
                                        double ratio_thre, bool show) {
    (void)show;
    return match_common(ESFM_KIND_F32X64, "SURF", cur_frame_1, cur_frame_2, matches, ratio_thre);
}

}  // namespace p3dv
