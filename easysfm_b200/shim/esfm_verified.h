// esfm_verified.h -- the verified match batch the two drop-in files share: p3dv::esfm_verify_all_pairs (feature_matching_gpu.cpp) fills it,
// MotionEstimator::estimate2D2D_E5P_RANSAC (estimate_motion_gpu.cpp) answers from it.  Header-only (one object through an inline function),
// so either file still builds and links on its own.
#ifndef ESFM_SHIM_VERIFIED_H_
#define ESFM_SHIM_VERIFIED_H_
#include <cstdint>
#include <cstdlib>
#include <unordered_map>
#include <vector>

#include "esfm_match.h"

namespace p3dv {
namespace esfm_shim {

struct VerifiedBatch {
    esfm_results_t* matches = nullptr;            // the prepared / loaded batch (owned by feature_matching_gpu.cpp)
    esfm_results_t* inliers = nullptr;            // its inlier matches, same pairs in the same order (owned here)
    std::vector<esfm_two_view_t> tv;              // one per pair
    std::unordered_map<uint64_t, int64_t> index;  // (query << 32 | train) -> first position in the batch
    double ransac_thre = 0.0, ransac_prob = 0.0;
    int min_pair = 0;                             // pairs with at most this many matches were not verified
    void clear() {
        if (inliers) esfm_results_destroy(inliers);
        inliers = nullptr;
        matches = nullptr;
        tv.clear();
        index.clear();
    }
    ~VerifiedBatch() { clear(); }
};

inline VerifiedBatch& verified() {
    static VerifiedBatch v;
    return v;
}

// $ESFM_RANSAC_SEED: the sampler seed of every two-view call, per call or batched
inline uint64_t ransac_seed() {
    const char* s = std::getenv("ESFM_RANSAC_SEED");
    return s ? std::strtoull(s, nullptr, 10) : 0;
}

}  // namespace esfm_shim
}  // namespace p3dv
#endif
