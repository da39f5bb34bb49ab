// tracks.cu -- SURVEY 8f rank 3: what consumes the pair matches right after the matching hot path.
//
//   * unique-id propagation over the pair loop (cpp_code/test/sfm.cpp:140-217): inherently sequential -- frame i's labels depend on
//     every earlier pair in loop order -- so it stays on the host, but in O(matches) instead of the reference's
//     O(matches x keypoints): the "is this id already used in frame i" linear scan (:178-185) becomes a hash lookup
//     (within a frame every non-negative id occurs at most once, because an id is only ever assigned when absent).
//   * initial frame pair (cpp_code/src/feature_matching.cpp:160-233): for EVERY pair the sum, over the points both frames see, of
//     the number of frames seeing the point.  The reference walks a dense frames x points bool matrix per pair
//     (O(N^2 P): 4e12 steps at 1000 frames x 8000 keypoints); here it is a CUDA kernel over sorted per-frame id lists:
//     one CTA holds frame i's list in shared memory and binary-searches the lists of a chunk of frames j < i against it.
//   * next frame (feature_matching.cpp:235-268): host, binary search in the sorted lists.
// Integer work throughout; bit-exact against the literal restatement in oracle/tracks_oracle.c (tests/test_tracks.py).
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <new>
#include <unordered_map>

#include "host_internal.h"

using namespace esfm;

struct esfm_tracks {
    int n_frames = 0;
    std::vector<int32_t> kp;                 // keypoints per frame
    std::vector<int64_t> kp_off;             // frame f's keypoints start here
    std::vector<int32_t> ids;                // frame_t::unique_pixel_ids, frames back to back (-1 = not labelled yet)
    std::vector<uint8_t> has_match;          // frame_t::unique_pixel_has_match
    std::vector<int32_t> sorted_ids;         // per finished frame: its ids ascending (same layout as ids)
    std::vector<int32_t> point_frames;       // per unique point: how many frames see it (point_track_frame_num, feature_matching.cpp:176)
    int frames_done = 0;                     // frames [0, frames_done) are finished
    int last_j = -1;                         // last train frame fed for the frame in progress
    int64_t n_points = 0;                    // cur_num_unique_points (sfm.cpp:138)
    std::unordered_map<int32_t, int32_t> present;   // frame in progress: id -> keypoint holding it
    // device copies for the scoring kernel (rebuilt when stale)
    esfm_ctx* dev_ctx = nullptr;
    int32_t* d_sorted = nullptr;
    int32_t* d_point_frames = nullptr;
    long long* d_kp_off = nullptr;
    long long* d_scores = nullptr;
    int dev_frames = -1;
};

namespace {

constexpr int kCovThreads = 256;
constexpr int kCovJChunk = 8;            // frames j handled by one CTA against the same frame i

// scores[i (i - 1) / 2 + j] = sum over ids present in both frames of point_frames[id]     (feature_matching.cpp:201-207)
__global__ void __launch_bounds__(kCovThreads) covis_score_kernel(const int32_t* __restrict__ sorted_ids, const long long* __restrict__ kp_off,
                                                                  const int32_t* __restrict__ point_frames, int n_frames, int smem_ids,
                                                                  long long* __restrict__ scores) {
    extern __shared__ int32_t s_ids[];
    __shared__ long long s_part[kCovThreads / 32];
    const int i = blockIdx.x;
    const int j0 = blockIdx.y * kCovJChunk;
    if (j0 >= i) return;
    const int32_t* li = sorted_ids + kp_off[i];
    const int ni = (int)(kp_off[i + 1] - kp_off[i]);
    const bool in_smem = ni <= smem_ids;
    if (in_smem)
        for (int e = threadIdx.x; e < ni; e += kCovThreads) s_ids[e] = li[e];
    __syncthreads();
    const int32_t* hay = in_smem ? s_ids : li;
    for (int j = j0; j < min(i, j0 + kCovJChunk); ++j) {
        const int32_t* lj = sorted_ids + kp_off[j];
        const int nj = (int)(kp_off[j + 1] - kp_off[j]);
        long long acc = 0;
        for (int e = threadIdx.x; e < nj; e += kCovThreads) {
            const int32_t id = lj[e];
            int lo = 0, hi = ni;                 // first position with hay[pos] >= id
            while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                if (hay[mid] < id) lo = mid + 1; else hi = mid;
            }
            if (lo < ni && hay[lo] == id) acc += point_frames[id];
        }
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, d);
        if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = acc;
        __syncthreads();
        if (threadIdx.x == 0) {
            long long tot = 0;
            for (int w = 0; w < kCovThreads / 32; ++w) tot += s_part[w];
            scores[(long long)i * (i - 1) / 2 + j] = tot;
        }
        __syncthreads();
    }
}

void free_device(esfm_tracks* t) {
    if (!t->dev_ctx) return;
    cudaSetDevice(t->dev_ctx->device);
    cudaFree(t->d_sorted); cudaFree(t->d_point_frames); cudaFree(t->d_kp_off); cudaFree(t->d_scores);
    t->d_sorted = nullptr; t->d_point_frames = nullptr; t->d_kp_off = nullptr; t->d_scores = nullptr;
    t->dev_ctx = nullptr;
    t->dev_frames = -1;
}

}  // namespace

extern "C" int esfm_tracks_create(int n_frames, const int32_t* keypoints_per_frame, esfm_tracks_t** out) {
    if (!out || (n_frames > 0 && !keypoints_per_frame) || n_frames < 0) return fail(ESFM_ERR_INVALID, "esfm_tracks_create: bad argument");
    *out = nullptr;
    esfm_tracks* t = new (std::nothrow) esfm_tracks();
    if (!t) return fail(ESFM_ERR_NOMEM, "out of host memory");
    t->n_frames = n_frames;
    t->kp.assign(keypoints_per_frame, keypoints_per_frame + n_frames);
    t->kp_off.assign((size_t)n_frames + 1, 0);
    for (int f = 0; f < n_frames; ++f) {
        if (t->kp[(size_t)f] < 0) { delete t; return fail(ESFM_ERR_INVALID, "frame %d has a negative keypoint count", f); }
        t->kp_off[(size_t)f + 1] = t->kp_off[(size_t)f] + t->kp[(size_t)f];
    }
    if (t->kp_off[(size_t)n_frames] > 0x7fffffffLL) { delete t; return fail(ESFM_ERR_CAPACITY, "more than 2^31 keypoints in total (ids are int, utility.h:33)"); }
    t->ids.assign((size_t)t->kp_off[(size_t)n_frames], -1);          // utility.h:44-51 init_pixel_ids
    t->has_match.assign(t->ids.size(), 0);
    t->sorted_ids.assign(t->ids.size(), 0);
    *out = t;
    return ESFM_OK;
}

extern "C" int esfm_tracks_destroy(esfm_tracks_t* t) {
    if (!t) return ESFM_OK;
    free_device(t);
    delete t;
    return ESFM_OK;
}

// sfm.cpp:172-194 for one pair (frame i in progress, frame j < i finished), matches in the caller's order.
extern "C" int esfm_tracks_add_pair(esfm_tracks_t* t, int frame_i, int frame_j, const esfm_dmatch_t* m, int n) {
    if (!t || (n > 0 && !m) || n < 0) return fail(ESFM_ERR_INVALID, "esfm_tracks_add_pair: bad argument");
    if (frame_i != t->frames_done || frame_i >= t->n_frames)
        return fail(ESFM_ERR_STATE, "pairs must arrive in the reference's loop order: frame %d is in progress, got %d", t->frames_done, frame_i);
    if (frame_j <= t->last_j || frame_j >= frame_i)
        return fail(ESFM_ERR_STATE, "pair (%d,%d): train frames must ascend below the query frame (last was %d)", frame_i, frame_j, t->last_j);
    t->last_j = frame_j;
    int32_t* idi = t->ids.data() + t->kp_off[(size_t)frame_i];
    const int32_t* idj = t->ids.data() + t->kp_off[(size_t)frame_j];
    uint8_t* hm = t->has_match.data() + t->kp_off[(size_t)frame_i];
    const int ni = t->kp[(size_t)frame_i], nj = t->kp[(size_t)frame_j];
    for (int k = 0; k < n; ++k) {
        const int q = m[k].queryIdx, tr = m[k].trainIdx;
        if (q < 0 || q >= ni || tr < 0 || tr >= nj)
            return fail(ESFM_ERR_INVALID, "pair (%d,%d): match %d = (%d,%d) is outside the frames' %d x %d keypoints", frame_i, frame_j, k, q, tr, ni, nj);
        const int32_t cand = idj[tr];                         // (>= 0: frame j is finished)
        if (idi[q] < 0 || idi[q] != cand) {                   // sfm.cpp:174-175
            if (t->present.find(cand) == t->present.end()) {  // :178-185, the linear duplicate scan as a lookup
                if (idi[q] >= 0) t->present.erase(idi[q]);    // the id this keypoint held leaves the frame
                idi[q] = cand;                                // :188
                hm[q] = 1;                                    // :189
                t->present.emplace(cand, q);
            }
        }
    }
    return ESFM_OK;
}

// sfm.cpp:199-213: fresh ids for the keypoints no pair labelled, the frame's row of the track matrix.
extern "C" int esfm_tracks_finish_frame(esfm_tracks_t* t, int frame_i) {
    if (!t) return fail(ESFM_ERR_INVALID, "tracks is NULL");
    if (frame_i != t->frames_done || frame_i >= t->n_frames) return fail(ESFM_ERR_STATE, "frame %d is in progress, got %d", t->frames_done, frame_i);
    int32_t* idi = t->ids.data() + t->kp_off[(size_t)frame_i];
    const int ni = t->kp[(size_t)frame_i];
    int64_t fresh = 0;
    for (int k = 0; k < ni; ++k)
        if (idi[k] < 0) { idi[k] = (int32_t)(t->n_points + fresh); ++fresh; }
    t->n_points += fresh;
    if ((size_t)t->n_points > t->point_frames.size()) t->point_frames.resize((size_t)t->n_points, 0);
    int32_t* si = t->sorted_ids.data() + t->kp_off[(size_t)frame_i];
    std::copy(idi, idi + ni, si);
    std::sort(si, si + ni);
    for (int k = 0; k < ni; ++k) t->point_frames[(size_t)si[k]] += 1;      // (ids are unique inside a frame)
    t->present.clear();
    t->last_j = -1;
    t->frames_done += 1;
    return ESFM_OK;
}

// The whole pair loop of sfm.cpp:140-217 over a batch that holds all pairs in the reference's order.  Pairs with at most
// `min_pair_matches` matches contribute nothing (sfm.cpp:163: `if (temp_matches.size() > num_min_pair)`, 20 in the reference);
// the others contribute ALL their matches.  The reference feeds the inliers of its 5-point RANSAC (estimate_motion.cpp:27-97): that is
// this loop over the batch esfm_two_view_results returns (pairs at or below 20 matches have no inliers there) with min_pair_matches = 0.
extern "C" int esfm_tracks_build(esfm_tracks_t* t, esfm_results_t* r, int min_pair_matches) {
    if (!t || !r) return fail(ESFM_ERR_INVALID, "esfm_tracks_build: NULL argument");
    if (t->frames_done != 0) return fail(ESFM_ERR_STATE, "tracks already (partly) built");
    int64_t n_pairs = 0;
    if (int rc = esfm_results_counts(r, &n_pairs, nullptr)) return rc;
    if (n_pairs != (int64_t)t->n_frames * (t->n_frames - 1) / 2)
        return fail(ESFM_ERR_INVALID, "the batch has %lld pairs, %d frames need %lld", (long long)n_pairs, t->n_frames, (long long)t->n_frames * (t->n_frames - 1) / 2);
    int64_t k = 0;
    for (int i = 0; i < t->n_frames; ++i) {
        for (int j = 0; j < i; ++j, ++k) {
            int q = -1, tr = -1, n = 0;
            const esfm_dmatch_t* m = nullptr;
            if (int rc = esfm_results_pair_at(r, k, &q, &tr, &m, &n)) return rc;
            if (q != i || tr != j) return fail(ESFM_ERR_INVALID, "pair %lld of the batch is (%d,%d), the loop order wants (%d,%d)", (long long)k, q, tr, i, j);
            if (n > min_pair_matches)
                if (int rc = esfm_tracks_add_pair(t, i, j, m, n)) return rc;
        }
        if (int rc = esfm_tracks_finish_frame(t, i)) return rc;
    }
    return ESFM_OK;
}

extern "C" int esfm_tracks_frame(esfm_tracks_t* t, int frame, const int32_t** unique_pixel_ids, const uint8_t** unique_pixel_has_match, int* n) {
    if (!t) return fail(ESFM_ERR_INVALID, "tracks is NULL");
    if (frame < 0 || frame >= t->n_frames) return fail(ESFM_ERR_INVALID, "frame %d out of range [0,%d)", frame, t->n_frames);
    if (unique_pixel_ids) *unique_pixel_ids = t->ids.data() + t->kp_off[(size_t)frame];
    if (unique_pixel_has_match) *unique_pixel_has_match = t->has_match.data() + t->kp_off[(size_t)frame];
    if (n) *n = t->kp[(size_t)frame];
    return ESFM_OK;
}

extern "C" int esfm_tracks_counts(esfm_tracks_t* t, int* frames_done, int64_t* n_unique_points) {
    if (!t) return fail(ESFM_ERR_INVALID, "tracks is NULL");
    if (frames_done) *frames_done = t->frames_done;
    if (n_unique_points) *n_unique_points = t->n_points;
    return ESFM_OK;
}

// Co-visibility score of every pair (i, j < i) in loop order, on the device.
extern "C" int esfm_tracks_pair_scores(esfm_ctx_t* ctx, esfm_tracks_t* t, int64_t* scores, double* kernel_ms) {
    if (!ctx || !t || !scores) return fail(ESFM_ERR_INVALID, "esfm_tracks_pair_scores: NULL argument");
    if (t->frames_done != t->n_frames) return fail(ESFM_ERR_STATE, "tracks are not finished (%d of %d frames)", t->frames_done, t->n_frames);
    const int n = t->n_frames;
    const int64_t n_pairs = (int64_t)n * (n - 1) / 2;
    if (kernel_ms) *kernel_ms = 0.0;
    if (n_pairs == 0) return ESFM_OK;
    CUDA_TRY(cudaSetDevice(ctx->device));
    if (t->dev_ctx != ctx || t->dev_frames != n) {
        free_device(t);
        t->dev_ctx = ctx;
        CUDA_TRY(cudaMalloc((void**)&t->d_sorted, std::max<size_t>(t->sorted_ids.size(), 1) * sizeof(int32_t)));
        CUDA_TRY(cudaMalloc((void**)&t->d_point_frames, std::max<size_t>(t->point_frames.size(), 1) * sizeof(int32_t)));
        CUDA_TRY(cudaMalloc((void**)&t->d_kp_off, ((size_t)n + 1) * sizeof(long long)));
        CUDA_TRY(cudaMalloc((void**)&t->d_scores, (size_t)n_pairs * sizeof(long long)));
        CUDA_TRY(cudaMemcpyAsync(t->d_sorted, t->sorted_ids.data(), t->sorted_ids.size() * sizeof(int32_t), cudaMemcpyHostToDevice, ctx->stream));
        CUDA_TRY(cudaMemcpyAsync(t->d_point_frames, t->point_frames.data(), t->point_frames.size() * sizeof(int32_t), cudaMemcpyHostToDevice, ctx->stream));
        static_assert(sizeof(long long) == sizeof(int64_t), "offset layout");
        CUDA_TRY(cudaMemcpyAsync(t->d_kp_off, t->kp_off.data(), ((size_t)n + 1) * sizeof(long long), cudaMemcpyHostToDevice, ctx->stream));
        ctx->stats.h2d_bytes += (t->sorted_ids.size() + t->point_frames.size()) * 4 + ((size_t)n + 1) * 8;
        t->dev_frames = n;
    }
    const int max_kp = *std::max_element(t->kp.begin(), t->kp.end());
    const int smem_ids = std::min(max_kp, 200 * 1024 / 4);         // larger frames are searched in global memory
    const size_t smem = (size_t)smem_ids * sizeof(int32_t);
    CUDA_TRY(cudaFuncSetAttribute(covis_score_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    ChunkBuf& cb = ctx->buf[0];
    CUDA_TRY(cudaEventRecord(cb.ev_t0, ctx->stream));
    const dim3 grid((unsigned)n, (unsigned)((n - 1 + kCovJChunk - 1) / kCovJChunk));
    covis_score_kernel<<<grid, kCovThreads, smem, ctx->stream>>>(t->d_sorted, t->d_kp_off, t->d_point_frames, n, smem_ids, t->d_scores);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaEventRecord(cb.ev_t1, ctx->stream));
    CUDA_TRY(cudaMemcpyAsync(scores, t->d_scores, (size_t)n_pairs * sizeof(long long), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    ctx->stats.kernel_launches += 1;
    ctx->stats.d2h_bytes += (size_t)n_pairs * 8;
    float ms = 0.f;
    CUDA_TRY(cudaEventElapsedTime(&ms, cb.ev_t0, cb.ev_t1));
    if (kernel_ms) *kernel_ms = ms;
    return ESFM_OK;
}

// feature_matching.cpp:160-233.  appro_depth[p] = img_match_graph[i][j].appro_depth in loop order (NULL: 1.0 everywhere, the value
// sfm.cpp:148 starts every pair with).  *found = 0 means no pair reached min_track_num_init: the reference then falls back to (1, 0).
extern "C" int esfm_tracks_find_init_pair(esfm_ctx_t* ctx, esfm_tracks_t* t, const double* appro_depth, int min_track_num_init,
                                          double max_depth_baseline_ratio_init, int* frame_1, int* frame_2, double* depth_init,
                                          int64_t* best_score, int* found) {
    if (!ctx || !t || !frame_1 || !frame_2) return fail(ESFM_ERR_INVALID, "esfm_tracks_find_init_pair: NULL argument");
    const int n = t->n_frames;
    const int64_t n_pairs = (int64_t)n * (n - 1) / 2;
    std::vector<int64_t> scores((size_t)n_pairs);
    if (int rc = esfm_tracks_pair_scores(ctx, t, scores.data(), nullptr)) return rc;
    int f1 = 0, f2 = 0;
    int64_t max_sum = min_track_num_init;                       // :188
    double ratio_init = 0.0;
    int64_t p = 0;
    for (int i = 0; i < n; ++i)
        for (int j = 0; j < i; ++j, ++p) {
            const double r = appro_depth ? appro_depth[p] : 1.0;
            if (r > max_depth_baseline_ratio_init) continue;    // :198-199
            if (scores[(size_t)p] >= max_sum) {                  // :208 ('>=': the last best pair in loop order wins)
                max_sum = scores[(size_t)p];
                ratio_init = r;
                f1 = i;
                f2 = j;
            }
        }
    const bool ok = f1 != f2;
    if (!ok) {                                                   // :219-226
        f1 = 1;
        f2 = 0;
        ratio_init = n > 1 ? (appro_depth ? appro_depth[0] : 1.0) : 0.0;
    }
    *frame_1 = f1;
    *frame_2 = f2;
    if (depth_init) *depth_init = ratio_init;
    if (best_score) *best_score = max_sum;
    if (found) *found = ok ? 1 : 0;
    return ESFM_OK;
}

// feature_matching.cpp:235-268: the unprocessed frame that sees most of the given 3D points ('>' : the first best frame wins;
// *next_frame is left untouched when no candidate sees any of them, as in the reference).
extern "C" int esfm_tracks_find_next_frame(esfm_tracks_t* t, const uint8_t* frames_to_process, const int32_t* point_ids, int64_t n_ids,
                                           int* next_frame, int* common_points) {
    if (!t || !frames_to_process || (n_ids > 0 && !point_ids) || !next_frame) return fail(ESFM_ERR_INVALID, "esfm_tracks_find_next_frame: NULL argument");
    if (t->frames_done != t->n_frames) return fail(ESFM_ERR_STATE, "tracks are not finished");
    int max_common = 0;
    for (int i = 0; i < t->n_frames; ++i) {
        if (!frames_to_process[i]) continue;
        const int32_t* si = t->sorted_ids.data() + t->kp_off[(size_t)i];
        const int ni = t->kp[(size_t)i];
        int common = 0;
        for (int64_t k = 0; k < n_ids; ++k) common += std::binary_search(si, si + ni, point_ids[k]) ? 1 : 0;
        if (common > max_common) { max_common = common; *next_frame = i; }
    }
    if (common_points) *common_points = max_common;
    return ESFM_OK;
}
