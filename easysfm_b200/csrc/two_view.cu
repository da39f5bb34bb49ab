// two_view.cu -- batched two-view geometric verification on the GPU matches (SURVEY 8f rank 1), sm_100a.
//
// Replaces, per image pair, the reference's
//     MotionEstimator::estimate2D2D_E5P_RANSAC   cpp_code/src/estimate_motion.cpp:27-97   (cv::findEssentialMat(RANSAC) :48-49, inlier
//                                                 matches :54-60, cv::recoverPose :65, T = [R t; 0 1] :72-82)
//     MotionEstimator::getDepthFast               cpp_code/src/estimate_motion.cpp:234-283 (cv::triangulatePoints, mean point norm)
// as called in the all-pairs loop at cpp_code/test/sfm.cpp:163-166.  The step is per-pair independent like the matching itself, so the same
// batch of pairs goes through four kernels (float64 throughout; the algorithms are those of two_view_math.cuh / oracle/two_view_oracle.py):
//   tv_normalise_kernel   pixel coordinates -> K^-1 x
//   tv_solve_kernel       one thread per (pair, hypothesis of the round): 5 matches from the counter-based sampler, Nister's minimal solver
//   tv_score_kernel       one warp per (pair, hypothesis): Sampson inliers of each of its <= 10 models over all matches of the pair
//   tv_select_kernel      one thread per pair: OpenCV's sequential RANSAC rule (first model with more inliers wins, adaptive iteration count)
//                         replayed over the round's counts -- the result is that of the sequential loop, hypothesis by hypothesis
//   tv_pose_kernel        one block per pair: inlier mask of the best model, the four (R, t) of the SVD, cheirality counts with DLT
//                         triangulation (recoverPose), mean depth of every random_rate-th inlier (getDepthFast)
// Rounds of kTvRound hypotheses repeat until max_iters; pairs whose stopping rule has fired skip the later rounds.
// esfm_two_view_results verifies a results batch with the same kernels: tv_gather_kernel takes the place of the host gather and
// tv_normalise_kernel, each pair draws its hypotheses from its frame ids, and tv_scan_kernel + tv_compact_kernel keep the inlier records on
// the device, so only they and the per-pair results cross back to the host.
#include <algorithm>
#include <new>
#include <vector>

#include "esfm_internal.cuh"
#include "host_internal.h"
#include "two_view_math.cuh"

namespace esfm {

namespace {

constexpr int kTvRound = 64;           // hypotheses per round and pair (the stopping rule fires after ~65 on typical pairs: 128 wasted half of round 1)
constexpr int kTvPoseThreads = 128;

struct TvState {                       // per pair, device
    double E[9];
    int best_count, niters, it, done;
};

__global__ void tv_normalise_kernel(const float* __restrict__ p1, const float* __restrict__ p2, const double* __restrict__ K, int k_per_pair,
                                    const long long* __restrict__ pair_off, int n_pairs, double2* __restrict__ n1, double2* __restrict__ n2) {
    const int pair = blockIdx.x;
    const double* Kp = K + (k_per_pair ? (size_t)pair * 9 : 0);
    const double fx = Kp[0], fy = Kp[4], cx = Kp[2], cy = Kp[5];
    for (long long i = pair_off[pair] + threadIdx.x; i < pair_off[pair + 1]; i += blockDim.x) {
        n1[i] = make_double2(((double)p1[2 * i] - cx) / fx, ((double)p1[2 * i + 1] - cy) / fy);
        n2[i] = make_double2(((double)p2[2 * i] - cx) / fx, ((double)p2[2 * i + 1] - cy) / fy);
    }
}

// esfm_two_view_results: the matches of a results batch in, normalised coordinates out -- tv_normalise_kernel's arithmetic on the key points the
// records name, so both entry points feed the solver the same bytes.  One block per pair; an index outside its frame's key points leaves (0, 0)
// and lowers *bad to the pair (the first offending pair of the chunk).
__global__ void tv_gather_kernel(const esfm_dmatch_t* __restrict__ rec, const PairDesc* __restrict__ frames, const long long* __restrict__ kp_off,
                                 const float* __restrict__ kp_xy, const double* __restrict__ K, int k_per_pair, const long long* __restrict__ pair_off,
                                 double2* __restrict__ n1, double2* __restrict__ n2, int* __restrict__ bad) {
    const int pair = blockIdx.x;
    const double* Kp = K + (k_per_pair ? (size_t)pair * 9 : 0);
    const double fx = Kp[0], fy = Kp[4], cx = Kp[2], cy = Kp[5];
    const PairDesc pd = frames[pair];
    const long long q0 = kp_off[pd.q_frame], nq = kp_off[pd.q_frame + 1] - q0;
    const long long t0 = kp_off[pd.t_frame], nt = kp_off[pd.t_frame + 1] - t0;
    for (long long i = pair_off[pair] + threadIdx.x; i < pair_off[pair + 1]; i += blockDim.x) {
        const int q = rec[i].queryIdx, t = rec[i].trainIdx;
        if (q < 0 || q >= nq || t < 0 || t >= nt) {
            atomicMin(bad, pair);
            n1[i] = n2[i] = make_double2(0.0, 0.0);
            continue;
        }
        const float* a = kp_xy + 2 * (q0 + q);
        const float* b = kp_xy + 2 * (t0 + t);
        n1[i] = make_double2(((double)a[0] - cx) / fx, ((double)a[1] - cy) / fy);
        n2[i] = make_double2(((double)b[0] - cx) / fx, ((double)b[1] - cy) / fy);
    }
}

// Pairs with at most `skip_at_most` matches are done before the first round (ok = 0, iters = 0); esfm_two_view_batch passes 4: a minimal
// sample needs five matches.
__global__ void tv_init_kernel(TvState* st, const long long* __restrict__ pair_off, int n_pairs, int max_iters, int skip_at_most) {
    const int pair = blockIdx.x * blockDim.x + threadIdx.x;
    if (pair >= n_pairs) return;
    TvState s;
    for (int e = 0; e < 9; ++e) s.E[e] = 0.0;
    s.best_count = 4;                  // OpenCV: a model must beat MAX(maxGoodCount, modelPoints - 1)
    s.niters = max_iters;
    s.it = 0;
    s.done = (pair_off[pair + 1] - pair_off[pair]) <= skip_at_most ? 1 : 0;
    st[pair] = s;
}

// Sampler key of pair p: keys[p] when given (esfm_two_view_results: the pair's frame ids), else first_pair + p (esfm_two_view_batch).
__global__ void __launch_bounds__(kTvRound) tv_solve_kernel(const double2* __restrict__ n1, const double2* __restrict__ n2, const long long* __restrict__ pair_off,
                                                             const TvState* __restrict__ st, int round, unsigned long long seed, unsigned long long first_pair,
                                                             const unsigned long long* __restrict__ keys, double* __restrict__ models, int* __restrict__ n_models) {
    const int pair = blockIdx.x;
    const TvState s = st[pair];
    const int hyp = round * kTvRound + threadIdx.x;
    int* nm = n_models + (size_t)pair * kTvRound + threadIdx.x;
    if (s.done || hyp >= s.niters) { *nm = 0; return; }
    const long long o = pair_off[pair];
    const unsigned m = (unsigned)(pair_off[pair + 1] - o);
    int idx[5];
    tv::sample_indices(seed, keys ? keys[pair] : first_pair + (unsigned long long)pair, (unsigned long long)hyp, m, idx);
    double q1[5][2], q2[5][2], Es[10][9];
    for (int k = 0; k < 5; ++k) {
        const double2 a = n1[o + idx[k]], b = n2[o + idx[k]];
        q1[k][0] = a.x; q1[k][1] = a.y; q2[k][0] = b.x; q2[k][1] = b.y;
    }
    const int n = tv::five_point(q1, q2, Es);
    double* out = models + ((size_t)pair * kTvRound + threadIdx.x) * 90;
    for (int k = 0; k < n; ++k)
        for (int e = 0; e < 9; ++e) out[9 * k + e] = Es[k][e];
    *nm = n;
}

__global__ void __launch_bounds__(256) tv_score_kernel(const double2* __restrict__ n1, const double2* __restrict__ n2, const long long* __restrict__ pair_off,
                                                        const double* __restrict__ K, int k_per_pair, double thre, const double* __restrict__ models,
                                                        const int* __restrict__ n_models, int* __restrict__ counts) {
    const int pair = blockIdx.y;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int h = blockIdx.x * 8 + warp;                       // hypothesis of the round
    const int n = n_models[(size_t)pair * kTvRound + h];
    if (n == 0) return;
    const double* Kp = K + (k_per_pair ? (size_t)pair * 9 : 0);
    const double tn = thre / ((Kp[0] + Kp[4]) * 0.5);
    const double t2 = tn * tn;
    const long long o = pair_off[pair];
    const int m = (int)(pair_off[pair + 1] - o);
    const double* Eb = models + ((size_t)pair * kTvRound + h) * 90;
    for (int k = 0; k < n; ++k) {
        double E[9];
#pragma unroll
        for (int e = 0; e < 9; ++e) E[e] = Eb[9 * k + e];
        int c = 0;
        for (int i = lane; i < m; i += 32) {
            const double2 a = n1[o + i], b = n2[o + i];
            c += tv::sampson_error(E, a.x, a.y, b.x, b.y) <= t2 ? 1 : 0;
        }
        c = __reduce_add_sync(0xffffffffu, c);
        if (lane == 0) counts[((size_t)pair * kTvRound + h) * 10 + k] = c;
    }
}

__global__ void tv_select_kernel(TvState* st, const long long* __restrict__ pair_off, int n_pairs, int round, double prob, const double* __restrict__ models,
                                 const int* __restrict__ n_models, const int* __restrict__ counts) {
    const int pair = blockIdx.x * blockDim.x + threadIdx.x;
    if (pair >= n_pairs) return;
    TvState s = st[pair];
    if (s.done) return;
    const int m = (int)(pair_off[pair + 1] - pair_off[pair]);
    for (int h = 0; h < kTvRound; ++h) {
        if (s.it >= s.niters) { s.done = 1; break; }
        const int n = n_models[(size_t)pair * kTvRound + h];
        for (int k = 0; k < n; ++k) {
            const int c = counts[((size_t)pair * kTvRound + h) * 10 + k];
            if (c > s.best_count) {
                s.best_count = c;
                const double* E = models + ((size_t)pair * kTvRound + h) * 90 + 9 * k;
                for (int e = 0; e < 9; ++e) s.E[e] = E[e];
                s.niters = tv::ransac_update_num_iters(prob, (double)(m - c) / m, 5, s.niters);
            }
        }
        ++s.it;
    }
    if (s.it >= s.niters) s.done = 1;
    st[pair] = s;
}

__device__ __forceinline__ int block_sum_int(int v, int* sh) {
    v = __reduce_add_sync(0xffffffffu, v);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
    __syncthreads();
    int t = 0;
    for (int w = 0; w < kTvPoseThreads / 32; ++w) t += sh[w];
    return t;
}

__global__ void __launch_bounds__(kTvPoseThreads) tv_pose_kernel(const double2* __restrict__ n1, const double2* __restrict__ n2, const long long* __restrict__ pair_off,
                                                                  const double* __restrict__ K, int k_per_pair, double thre, double dist, int random_rate,
                                                                  const TvState* __restrict__ st, unsigned char* __restrict__ mask, esfm_two_view_t* __restrict__ out) {
    const int pair = blockIdx.x;
    const long long o = pair_off[pair];
    const int m = (int)(pair_off[pair + 1] - o);
    const TvState s = st[pair];
    __shared__ int sh_i[kTvPoseThreads / 32];
    __shared__ double sh_R[4][9], sh_t[4][3], sh_d[kTvPoseThreads];
    __shared__ int sh_pick;
    const bool ok = s.best_count > 4;
    const double* Kp = K + (k_per_pair ? (size_t)pair * 9 : 0);
    const double tn = thre / ((Kp[0] + Kp[4]) * 0.5);
    const double t2 = tn * tn;
    // inlier mask of the best model
    int cnt = 0;
    for (int i = threadIdx.x; i < m; i += kTvPoseThreads) {
        unsigned char f = 0;
        if (ok) {
            const double2 a = n1[o + i], b = n2[o + i];
            f = tv::sampson_error(s.E, a.x, a.y, b.x, b.y) <= t2 ? 1 : 0;
        }
        mask[o + i] = f;
        cnt += f;
    }
    const int n_inl = block_sum_int(cnt, sh_i);
    esfm_two_view_t r;
    for (int e = 0; e < 9; ++e) { r.E[e] = ok ? s.E[e] : 0.0; r.R[e] = 0.0; }
    r.t[0] = r.t[1] = r.t[2] = 0.0;
    r.depth = 0.0;
    r.n_matches = m; r.n_inliers = n_inl; r.n_good = 0; r.iters = s.it; r.ok = ok ? 1 : 0; r.reserved = 0;
    if (!ok) {
        if (threadIdx.x == 0) out[pair] = r;
        return;
    }
    // recoverPose: the four candidates (R1, t), (R2, t), (R1, -t), (R2, -t)
    if (threadIdx.x == 0) {
        double R1[9], R2[9], t[3];
        tv::decompose_essential(s.E, R1, R2, t);
        for (int e = 0; e < 9; ++e) { sh_R[0][e] = R1[e]; sh_R[1][e] = R2[e]; sh_R[2][e] = R1[e]; sh_R[3][e] = R2[e]; }
        for (int e = 0; e < 3; ++e) { sh_t[0][e] = t[e]; sh_t[1][e] = t[e]; sh_t[2][e] = -t[e]; sh_t[3][e] = -t[e]; }
    }
    __syncthreads();
    int good[4] = {0, 0, 0, 0};
    for (int i = threadIdx.x; i < m; i += kTvPoseThreads) {
        if (!mask[o + i]) continue;
        const double2 a = n1[o + i], b = n2[o + i];
#pragma unroll
        for (int c = 0; c < 4; ++c) good[c] += tv::cheirality_ok(sh_R[c], sh_t[c], a.x, a.y, b.x, b.y, dist) ? 1 : 0;
    }
    int g[4];
    for (int c = 0; c < 4; ++c) g[c] = block_sum_int(good[c], sh_i);
    if (threadIdx.x == 0) {
        int k;
        if (g[0] >= g[1] && g[0] >= g[2] && g[0] >= g[3]) k = 0;
        else if (g[1] >= g[0] && g[1] >= g[2] && g[1] >= g[3]) k = 1;
        else if (g[2] >= g[0] && g[2] >= g[1] && g[2] >= g[3]) k = 2;
        else k = 3;
        sh_pick = k;
    }
    __syncthreads();
    const int k = sh_pick;
    // getDepthFast: every random_rate-th inlier (in match order) triangulated with [I|0], [R|t]; mean point norm.  Deterministic: each thread
    // sums its own points in order, the partial sums are added in thread order.
    double acc = 0.0;
    int base = 0, used = 0;
    for (int i0 = 0; i0 < m; i0 += kTvPoseThreads) {
        const int i = i0 + threadIdx.x;
        const int f = (i < m && mask[o + i]) ? 1 : 0;
        // ordinal of this inlier among the pair's inliers
        const unsigned bal = __ballot_sync(0xffffffffu, f);
        __syncthreads();
        if ((threadIdx.x & 31) == 0) sh_i[threadIdx.x >> 5] = __popc(bal);
        __syncthreads();
        int before = 0, total = 0;
        for (int w = 0; w < kTvPoseThreads / 32; ++w) {
            const int c = sh_i[w];
            before += w < (int)(threadIdx.x >> 5) ? c : 0;
            total += c;
        }
        const int ord = base + before + __popc(bal & ((1u << (threadIdx.x & 31)) - 1u));
        if (f && ord % random_rate == 0) {
            const double2 a = n1[o + i], b = n2[o + i];
            double Q[4];
            tv::triangulate_dlt(sh_R[k], sh_t[k], a.x, a.y, b.x, b.y, Q);
            const double x = Q[0] / Q[3], y = Q[1] / Q[3], z = Q[2] / Q[3];
            acc += sqrt(x * x + y * y + z * z);
            ++used;
        }
        base += total;
    }
    sh_d[threadIdx.x] = acc;
    const int n_used = block_sum_int(used, sh_i);
    if (threadIdx.x == 0) {
        double sum = 0.0;
        for (int w = 0; w < kTvPoseThreads; ++w) sum += sh_d[w];
        for (int e = 0; e < 9; ++e) r.R[e] = sh_R[k][e];
        for (int e = 0; e < 3; ++e) r.t[e] = sh_t[k][e];
        r.n_good = g[k];
        r.depth = n_used > 0 ? sum / n_used : 0.0;
        out[pair] = r;
    }
}

// Exclusive scan of the chunk's per-pair inlier counts (n_pairs <= 4096: one block, a few consecutive pairs per thread); inl_off[n_pairs] = total.
constexpr int kTvScanThreads = 1024;
__global__ void __launch_bounds__(kTvScanThreads) tv_scan_kernel(const esfm_two_view_t* __restrict__ tv, int n_pairs, long long* __restrict__ inl_off) {
    __shared__ long long sh_w[kTvScanThreads / 32];
    const int per = (n_pairs + kTvScanThreads - 1) / kTvScanThreads;
    const int b = min(n_pairs, (int)threadIdx.x * per), e = min(n_pairs, b + per);
    long long v = 0;
    for (int p = b; p < e; ++p) v += tv[p].n_inliers;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    long long x = v;                                             // inclusive scan inside the warp
    for (int d = 1; d < 32; d <<= 1) {
        const long long y = __shfl_up_sync(0xffffffffu, x, d);
        if (lane >= d) x += y;
    }
    if (lane == 31) sh_w[warp] = x;
    __syncthreads();
    long long run = x - v;
    for (int w = 0; w < warp; ++w) run += sh_w[w];
    for (int p = b; p < e; ++p) { inl_off[p] = run; run += tv[p].n_inliers; }
    if (threadIdx.x == kTvScanThreads - 1) inl_off[n_pairs] = run;
}

// Stable compaction: the records of pair p whose mask is 1, in their order, to dst[inl_off[p] ...].  One block per pair, 128 matches at a time.
__global__ void __launch_bounds__(kTvPoseThreads) tv_compact_kernel(const esfm_dmatch_t* __restrict__ rec, const long long* __restrict__ pair_off,
                                                                     const unsigned char* __restrict__ mask, const long long* __restrict__ inl_off,
                                                                     esfm_dmatch_t* __restrict__ dst) {
    __shared__ int sh_w[kTvPoseThreads / 32];
    const int pair = blockIdx.x;
    if (inl_off[pair + 1] == inl_off[pair]) return;
    const long long o = pair_off[pair];
    const int m = (int)(pair_off[pair + 1] - o);
    long long base = inl_off[pair];
    for (int i0 = 0; i0 < m; i0 += kTvPoseThreads) {
        const int i = i0 + threadIdx.x;
        const int f = (i < m && mask[o + i]) ? 1 : 0;
        const unsigned bal = __ballot_sync(0xffffffffu, f);
        __syncthreads();
        if ((threadIdx.x & 31) == 0) sh_w[threadIdx.x >> 5] = __popc(bal);
        __syncthreads();
        int before = 0, total = 0;
        for (int w = 0; w < kTvPoseThreads / 32; ++w) {
            const int c = sh_w[w];
            before += w < (int)(threadIdx.x >> 5) ? c : 0;
            total += c;
        }
        if (f) dst[base + before + __popc(bal & ((1u << (threadIdx.x & 31)) - 1u))] = rec[o + i];
        base += total;
    }
}

// getDepthFast on its own (estimate_motion.cpp:234-283): every random_rate-th of the GIVEN matches triangulated with [I|0], [R|t]; mean norm.
// One block; deterministic summation (per-thread partial sums added in thread order).  Index, stride and n are 64-bit: random_rate may be
// anything up to INT_MAX, and threadIdx.x * random_rate or 128 * random_rate would wrap in 32 bits.
__global__ void __launch_bounds__(kTvPoseThreads) tv_depth_kernel(const float* __restrict__ p1, const float* __restrict__ p2, long long n,
                                                                   const double* __restrict__ K, const double* __restrict__ Rt, int random_rate,
                                                                   double* __restrict__ out) {
    __shared__ double sh_d[kTvPoseThreads];
    __shared__ long long sh_n[kTvPoseThreads];
    const double fx = K[0], fy = K[4], cx = K[2], cy = K[5];
    double acc = 0.0;
    long long used = 0;
    const long long stride = (long long)kTvPoseThreads * random_rate;
    for (long long i = (long long)threadIdx.x * random_rate; i < n; i += stride) {
        double Q[4];
        tv::triangulate_dlt(Rt, Rt + 9, ((double)p1[2 * i] - cx) / fx, ((double)p1[2 * i + 1] - cy) / fy, ((double)p2[2 * i] - cx) / fx,
                            ((double)p2[2 * i + 1] - cy) / fy, Q);
        const double x = Q[0] / Q[3], y = Q[1] / Q[3], z = Q[2] / Q[3];
        acc += sqrt(x * x + y * y + z * z);
        ++used;
    }
    sh_d[threadIdx.x] = acc;
    sh_n[threadIdx.x] = used;
    __syncthreads();
    if (threadIdx.x == 0) {
        double sum = 0.0;
        long long cnt = 0;
        for (int w = 0; w < kTvPoseThreads; ++w) { sum += sh_d[w]; cnt += sh_n[w]; }
        out[0] = cnt > 0 ? sum / cnt : 0.0;
        out[1] = (double)cnt;
    }
}

// device scratch of one call, from the context's private stream-ordered pool (freed blocks stay cached there: repeated calls do not
// allocate; cudaMalloc / cudaFree per call cost a third of a 2048-pair batch)
struct DevBuf {
    void* p = nullptr;
    esfm_ctx* ctx = nullptr;
    ~DevBuf() { if (p) cudaFreeAsync(p, ctx->stream); }
    cudaError_t alloc(esfm_ctx* c, size_t bytes) {
        ctx = c;
        return cudaMallocFromPoolAsync(&p, std::max<size_t>(bytes, 16), c->mempool, c->stream);
    }
    template <typename T> T* as() { return static_cast<T*>(p); }
};

bool bad_params(const esfm_two_view_params_t& p) { return p.max_iters < 1 || p.random_rate < 1 || !(p.ransac_thre > 0.0); }

constexpr int64_t kTvChunk = 4096;     // pairs per chunk: a round's hypotheses are kept for the whole chunk (64 x 10 models x 72 B a pair)
constexpr uint64_t kSegOffMask = ((uint64_t)1 << 40) - 1;

}  // namespace

}  // namespace esfm

using namespace esfm;

extern "C" int esfm_two_view_default_params(esfm_two_view_params_t* p) {
    if (!p) return fail(ESFM_ERR_INVALID, "esfm_two_view_default_params: NULL argument");
    p->ransac_thre = 1.0;          // estimate_motion.h:20
    p->ransac_prob = 0.99;
    p->max_iters = 1000;           // cv::findEssentialMat's default
    p->random_rate = 1;
    p->seed = 0;
    p->first_pair = 0;
    p->cheirality_dist = 50.0;     // cv::recoverPose's distanceThresh
    return ESFM_OK;
}

extern "C" int esfm_two_view_batch(esfm_ctx_t* ctx, int64_t n_pairs, const int64_t* pair_off, const float* pts1, const float* pts2, const double* K,
                                   int k_per_pair, const esfm_two_view_params_t* params, unsigned char* inlier_mask, esfm_two_view_t* out) {
    if (!ctx || !pair_off || !K || !params || !out || n_pairs < 0) return fail(ESFM_ERR_INVALID, "esfm_two_view_batch: NULL argument");
    if (bad_params(*params)) return fail(ESFM_ERR_INVALID, "esfm_two_view_batch: bad parameters");
    if (int rc = set_device(ctx)) return rc;
    if (n_pairs == 0) return ESFM_OK;
    for (int64_t p = 0; p < n_pairs; ++p)
        if (pair_off[p + 1] < pair_off[p]) return fail(ESFM_ERR_INVALID, "esfm_two_view_batch: pair_off must be non-decreasing");
    if (pair_off[0] != 0) return fail(ESFM_ERR_INVALID, "esfm_two_view_batch: pair_off[0] must be 0");
    const int64_t total = pair_off[n_pairs];
    if (total > 0 && (!pts1 || !pts2 || !inlier_mask)) return fail(ESFM_ERR_INVALID, "esfm_two_view_batch: NULL point arrays");
    cudaStream_t s = ctx->stream;
    const int64_t chunk = kTvChunk;
    DevBuf d_p1, d_p2, d_n1, d_n2, d_K, d_off, d_models, d_nm, d_counts, d_state, d_mask, d_out;
    const int64_t max_pairs = std::min<int64_t>(chunk, n_pairs);
    int64_t max_pts = 0;
    for (int64_t c0 = 0; c0 < n_pairs; c0 += chunk) max_pts = std::max<int64_t>(max_pts, pair_off[std::min(n_pairs, c0 + chunk)] - pair_off[c0]);
    CUDA_TRY(d_p1.alloc(ctx, (size_t)max_pts * 8)); CUDA_TRY(d_p2.alloc(ctx, (size_t)max_pts * 8));
    CUDA_TRY(d_n1.alloc(ctx, (size_t)max_pts * 16)); CUDA_TRY(d_n2.alloc(ctx, (size_t)max_pts * 16));
    CUDA_TRY(d_K.alloc(ctx, (size_t)(k_per_pair ? max_pairs : 1) * 72)); CUDA_TRY(d_off.alloc(ctx, (size_t)(max_pairs + 1) * 8));
    CUDA_TRY(d_models.alloc(ctx, (size_t)max_pairs * kTvRound * 90 * 8)); CUDA_TRY(d_nm.alloc(ctx, (size_t)max_pairs * kTvRound * 4));
    CUDA_TRY(d_counts.alloc(ctx, (size_t)max_pairs * kTvRound * 10 * 4)); CUDA_TRY(d_state.alloc(ctx, (size_t)max_pairs * sizeof(TvState)));
    CUDA_TRY(d_mask.alloc(ctx, (size_t)max_pts)); CUDA_TRY(d_out.alloc(ctx, (size_t)max_pairs * sizeof(esfm_two_view_t)));
    std::vector<long long> off;
    const int rounds = (params->max_iters + kTvRound - 1) / kTvRound;
    for (int64_t c0 = 0; c0 < n_pairs; c0 += chunk) {
        const int np = (int)std::min<int64_t>(chunk, n_pairs - c0);
        const int64_t p0 = pair_off[c0], npts = pair_off[c0 + np] - p0;
        off.resize((size_t)np + 1);
        for (int p = 0; p <= np; ++p) off[(size_t)p] = (long long)(pair_off[c0 + p] - p0);
        CUDA_TRY(cudaMemcpyAsync(d_off.p, off.data(), (size_t)(np + 1) * 8, cudaMemcpyHostToDevice, s));
        if (npts > 0) {
            CUDA_TRY(cudaMemcpyAsync(d_p1.p, pts1 + 2 * p0, (size_t)npts * 8, cudaMemcpyHostToDevice, s));
            CUDA_TRY(cudaMemcpyAsync(d_p2.p, pts2 + 2 * p0, (size_t)npts * 8, cudaMemcpyHostToDevice, s));
        }
        CUDA_TRY(cudaMemcpyAsync(d_K.p, K + (k_per_pair ? (size_t)c0 * 9 : 0), (size_t)(k_per_pair ? np : 1) * 72, cudaMemcpyHostToDevice, s));
        ctx->stats.h2d_bytes += (size_t)npts * 16 + (size_t)(np + 1) * 8;
        tv_normalise_kernel<<<np, 128, 0, s>>>(d_p1.as<float>(), d_p2.as<float>(), d_K.as<double>(), k_per_pair ? 1 : 0, d_off.as<long long>(), np,
                                               d_n1.as<double2>(), d_n2.as<double2>());
        tv_init_kernel<<<(np + 127) / 128, 128, 0, s>>>(d_state.as<TvState>(), d_off.as<long long>(), np, params->max_iters, 4);
        for (int r = 0; r < rounds; ++r) {
            tv_solve_kernel<<<np, kTvRound, 0, s>>>(d_n1.as<double2>(), d_n2.as<double2>(), d_off.as<long long>(), d_state.as<TvState>(), r,
                                                    (unsigned long long)params->seed, (unsigned long long)params->first_pair + (unsigned long long)c0,
                                                    nullptr, d_models.as<double>(), d_nm.as<int>());
            tv_score_kernel<<<dim3(kTvRound / 8, np), 256, 0, s>>>(d_n1.as<double2>(), d_n2.as<double2>(), d_off.as<long long>(), d_K.as<double>(), k_per_pair ? 1 : 0,
                                                                   params->ransac_thre, d_models.as<double>(), d_nm.as<int>(), d_counts.as<int>());
            tv_select_kernel<<<(np + 127) / 128, 128, 0, s>>>(d_state.as<TvState>(), d_off.as<long long>(), np, r, params->ransac_prob, d_models.as<double>(),
                                                              d_nm.as<int>(), d_counts.as<int>());
            ctx->stats.kernel_launches += 3;
        }
        tv_pose_kernel<<<np, kTvPoseThreads, 0, s>>>(d_n1.as<double2>(), d_n2.as<double2>(), d_off.as<long long>(), d_K.as<double>(), k_per_pair ? 1 : 0,
                                                     params->ransac_thre, params->cheirality_dist, params->random_rate, d_state.as<TvState>(),
                                                     d_mask.as<unsigned char>(), d_out.as<esfm_two_view_t>());
        ctx->stats.kernel_launches += 3;
        CUDA_TRY(cudaGetLastError());
        if (npts > 0) CUDA_TRY(cudaMemcpyAsync(inlier_mask + p0, d_mask.p, (size_t)npts, cudaMemcpyDeviceToHost, s));
        CUDA_TRY(cudaMemcpyAsync(out + c0, d_out.p, (size_t)np * sizeof(esfm_two_view_t), cudaMemcpyDeviceToHost, s));
        CUDA_TRY(cudaStreamSynchronize(s));
        ctx->stats.d2h_bytes += (size_t)npts + (size_t)np * sizeof(esfm_two_view_t);
    }
    return ESFM_OK;
}

extern "C" int esfm_two_view_depth(esfm_ctx_t* ctx, int64_t n_matches, const float* pts1, const float* pts2, const double* K, const double* R,
                                   const double* t, int random_rate, double* depth, int32_t* n_used) {
    if (!ctx || !K || !R || !t || !depth || n_matches < 0 || random_rate < 1) return fail(ESFM_ERR_INVALID, "esfm_two_view_depth: bad argument");
    if (n_matches > 0 && (!pts1 || !pts2)) return fail(ESFM_ERR_INVALID, "esfm_two_view_depth: NULL point arrays");
    if (int rc = set_device(ctx)) return rc;
    *depth = 0.0;
    if (n_used) *n_used = 0;
    if (n_matches == 0) return ESFM_OK;
    cudaStream_t s = ctx->stream;
    DevBuf d_p1, d_p2, d_par, d_out;
    CUDA_TRY(d_p1.alloc(ctx, (size_t)n_matches * 8)); CUDA_TRY(d_p2.alloc(ctx, (size_t)n_matches * 8)); CUDA_TRY(d_par.alloc(ctx, 21 * 8)); CUDA_TRY(d_out.alloc(ctx, 16));
    double par[21];
    for (int e = 0; e < 9; ++e) { par[e] = K[e]; par[9 + e] = R[e]; }
    for (int e = 0; e < 3; ++e) par[18 + e] = t[e];
    CUDA_TRY(cudaMemcpyAsync(d_p1.p, pts1, (size_t)n_matches * 8, cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaMemcpyAsync(d_p2.p, pts2, (size_t)n_matches * 8, cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaMemcpyAsync(d_par.p, par, sizeof par, cudaMemcpyHostToDevice, s));
    tv_depth_kernel<<<1, kTvPoseThreads, 0, s>>>(d_p1.as<float>(), d_p2.as<float>(), (long long)n_matches, d_par.as<double>(), d_par.as<double>() + 9, random_rate,
                                                 d_out.as<double>());
    CUDA_TRY(cudaGetLastError());
    double out[2];
    CUDA_TRY(cudaMemcpyAsync(out, d_out.p, 16, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    ctx->stats.kernel_launches += 1;
    *depth = out[0];
    if (n_used) *n_used = (int32_t)out[1];
    return ESFM_OK;
}

// ------------------------------------------------------------------------------------------------
// verification of a results batch: key points gathered, inliers compacted, on the device
// ------------------------------------------------------------------------------------------------
int esfm::two_view_job(const char* who, esfm_results* r, int n_frames, const int64_t* kp_off, const float* kp_xy, const double* K, int k_per_frame,
                       const esfm_two_view_params_t* params, int min_pair_matches, esfm_results_t** inliers, esfm_two_view_t* out, TvJob* job) {
    if (inliers) *inliers = nullptr;
    if (!r || !kp_off || !K || !params || !inliers || !out || n_frames < 0) return fail(ESFM_ERR_INVALID, "%s: NULL argument", who);
    if (!r->fetched) return fail(ESFM_ERR_STATE, "%s: matches are device-resident; call esfm_results_fetch first", who);
    if (r->keep == ESFM_KEEP_DIGESTS) return fail(ESFM_ERR_STATE, "%s: this batch kept per-pair digests only (ESFM_KEEP_DIGESTS)", who);
    if (bad_params(*params)) return fail(ESFM_ERR_INVALID, "%s: bad parameters", who);
    if (params->first_pair != 0) return fail(ESFM_ERR_INVALID, "%s: params->first_pair must be 0 (pairs are keyed by their frame ids)", who);
    if (kp_off[0] != 0) return fail(ESFM_ERR_INVALID, "%s: kp_off[0] must be 0", who);
    for (int f = 0; f < n_frames; ++f)
        if (kp_off[f + 1] < kp_off[f] || kp_off[f + 1] - kp_off[f] > INT32_MAX) return fail(ESFM_ERR_INVALID, "%s: kp_off must be non-decreasing (frame %d)", who, f);
    if (kp_off[n_frames] > 0 && !kp_xy) return fail(ESFM_ERR_INVALID, "%s: NULL key points", who);
    if (!r->frame_rows.empty()) {
        if ((int)r->frame_rows.size() != n_frames) return fail(ESFM_ERR_INVALID, "%s: the batch was matched on %zu frames, the caller has %d", who, r->frame_rows.size(), n_frames);
        for (int f = 0; f < n_frames; ++f)
            if ((int64_t)r->frame_rows[(size_t)f] != kp_off[f + 1] - kp_off[f])
                return fail(ESFM_ERR_INVALID, "%s: frame %d had %d descriptors when the batch was matched, it has %lld key points", who, f, r->frame_rows[(size_t)f],
                            (long long)(kp_off[f + 1] - kp_off[f]));
    }
    for (size_t k = 0; k < r->pairs.size(); ++k) {
        const int q = r->pairs[k].q_frame, t = r->pairs[k].t_frame;
        if (q < 0 || q >= n_frames || t < 0 || t >= n_frames) return fail(ESFM_ERR_INVALID, "%s: pair %zu = (%d,%d) is outside the caller's %d frames", who, k, q, t, n_frames);
    }
    job->matches = r;
    job->n_frames = n_frames;
    job->kp_off = kp_off;
    job->kp_xy = kp_xy;
    job->K = K;
    job->k_per_frame = k_per_frame ? 1 : 0;
    job->params = *params;
    job->min_pair_matches = min_pair_matches;
    return ESFM_OK;
}

// The share's pairs in chunks of <= 4096: their match records are uploaded from the batch's host segments (runs of consecutive pairs in one
// copy), gathered into normalised coordinates, verified by the kernels of esfm_two_view_batch with frame-id keys, and compacted; only the
// inlier records and the per-pair results come back.
int esfm::two_view_share(esfm_ctx* ctx, const TvJob& job, TvShare& sh) {
    const esfm_results* r = job.matches;
    const int64_t n = (int64_t)sh.ids.size();
    sh.counts.assign((size_t)n, 0);
    sh.offsets.assign((size_t)n, 0);
    sh.tv.resize((size_t)n);
    if (n == 0) return ESFM_OK;
    if (int rc = set_device(ctx)) return rc;
    cudaStream_t s = ctx->stream;
    const int64_t max_pairs = std::min<int64_t>(kTvChunk, n);
    int64_t max_pts = 0;
    for (int64_t c0 = 0; c0 < n; c0 += kTvChunk) {
        int64_t pts = 0;
        for (int64_t p = c0; p < std::min(n, c0 + kTvChunk); ++p) pts += r->counts[(size_t)sh.ids[(size_t)p]];
        max_pts = std::max(max_pts, pts);
    }
    const int64_t n_kp = job.kp_off[job.n_frames];
    DevBuf d_kp, d_kp_off, d_rec, d_n1, d_n2, d_K, d_off, d_frames, d_keys, d_models, d_nm, d_counts, d_state, d_mask, d_out, d_inl_off, d_inl, d_bad;
    CUDA_TRY(d_kp.alloc(ctx, (size_t)n_kp * 8)); CUDA_TRY(d_kp_off.alloc(ctx, (size_t)(job.n_frames + 1) * 8));
    CUDA_TRY(d_rec.alloc(ctx, (size_t)max_pts * sizeof(esfm_dmatch_t))); CUDA_TRY(d_inl.alloc(ctx, (size_t)max_pts * sizeof(esfm_dmatch_t)));
    CUDA_TRY(d_n1.alloc(ctx, (size_t)max_pts * 16)); CUDA_TRY(d_n2.alloc(ctx, (size_t)max_pts * 16)); CUDA_TRY(d_mask.alloc(ctx, (size_t)max_pts));
    CUDA_TRY(d_K.alloc(ctx, (size_t)(job.k_per_frame ? max_pairs : 1) * 72)); CUDA_TRY(d_off.alloc(ctx, (size_t)(max_pairs + 1) * 8));
    CUDA_TRY(d_frames.alloc(ctx, (size_t)max_pairs * sizeof(PairDesc))); CUDA_TRY(d_keys.alloc(ctx, (size_t)max_pairs * 8));
    CUDA_TRY(d_models.alloc(ctx, (size_t)max_pairs * kTvRound * 90 * 8)); CUDA_TRY(d_nm.alloc(ctx, (size_t)max_pairs * kTvRound * 4));
    CUDA_TRY(d_counts.alloc(ctx, (size_t)max_pairs * kTvRound * 10 * 4)); CUDA_TRY(d_state.alloc(ctx, (size_t)max_pairs * sizeof(TvState)));
    CUDA_TRY(d_out.alloc(ctx, (size_t)max_pairs * sizeof(esfm_two_view_t))); CUDA_TRY(d_inl_off.alloc(ctx, (size_t)(max_pairs + 1) * 8));
    CUDA_TRY(d_bad.alloc(ctx, 4));
    // key points and their offsets: once per call
    if (n_kp > 0) CUDA_TRY(cudaMemcpyAsync(d_kp.p, job.kp_xy, (size_t)n_kp * 8, cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaMemcpyAsync(d_kp_off.p, job.kp_off, (size_t)(job.n_frames + 1) * 8, cudaMemcpyHostToDevice, s));
    ctx->stats.h2d_bytes += (size_t)n_kp * 8 + (size_t)(job.n_frames + 1) * 8;
    const int rounds = (job.params.max_iters + kTvRound - 1) / kTvRound;
    const int skip_at_most = std::max(4, job.min_pair_matches);
    std::vector<long long> off, inl_off;
    std::vector<PairDesc> frames;
    std::vector<unsigned long long> keys;
    std::vector<double> Kc;
    for (int64_t c0 = 0; c0 < n; c0 += kTvChunk) {
        const int np = (int)std::min<int64_t>(kTvChunk, n - c0);
        off.assign((size_t)np + 1, 0);
        frames.resize((size_t)np);
        keys.resize((size_t)np);
        Kc.resize(job.k_per_frame ? (size_t)np * 9 : 9);
        for (int p = 0; p < np; ++p) {
            const size_t g = (size_t)sh.ids[(size_t)(c0 + p)];
            const PairDesc pd = r->pairs[g];
            off[(size_t)p + 1] = off[(size_t)p] + r->counts[g];
            frames[(size_t)p] = pd;
            keys[(size_t)p] = ((unsigned long long)(uint32_t)pd.q_frame << 32) | (uint32_t)pd.t_frame;
            if (job.k_per_frame) std::copy(job.K + (size_t)pd.q_frame * 9, job.K + (size_t)pd.q_frame * 9 + 9, Kc.begin() + (size_t)p * 9);   // the query frame's camera
        }
        if (!job.k_per_frame) std::copy(job.K, job.K + 9, Kc.begin());
        const int64_t npts = off[(size_t)np];
        CUDA_TRY(cudaMemcpyAsync(d_off.p, off.data(), (size_t)(np + 1) * 8, cudaMemcpyHostToDevice, s));
        CUDA_TRY(cudaMemcpyAsync(d_frames.p, frames.data(), (size_t)np * sizeof(PairDesc), cudaMemcpyHostToDevice, s));
        CUDA_TRY(cudaMemcpyAsync(d_keys.p, keys.data(), (size_t)np * 8, cudaMemcpyHostToDevice, s));
        CUDA_TRY(cudaMemcpyAsync(d_K.p, Kc.data(), Kc.size() * 8, cudaMemcpyHostToDevice, s));
        const int no_bad = INT32_MAX;
        CUDA_TRY(cudaMemcpyAsync(d_bad.p, &no_bad, 4, cudaMemcpyHostToDevice, s));
        // match records: consecutive pairs of one segment lie back to back, so a run of them is one copy
        const esfm_dmatch_t* run = nullptr;
        int64_t run_len = 0, run_dst = 0;
        for (int p = 0; p <= np; ++p) {
            const esfm_dmatch_t* src = nullptr;
            int64_t cnt = 0;
            if (p < np) {
                const size_t g = (size_t)sh.ids[(size_t)(c0 + p)];
                cnt = r->counts[g];
                if (cnt == 0) continue;
                const uint64_t o = r->offsets[g];
                src = r->segments[(size_t)(o >> 40)].ptr + (o & kSegOffMask);
                if (run && src == run + run_len) { run_len += cnt; continue; }
            }
            if (run_len > 0)
                CUDA_TRY(cudaMemcpyAsync(d_rec.as<esfm_dmatch_t>() + run_dst, run, (size_t)run_len * sizeof(esfm_dmatch_t), cudaMemcpyHostToDevice, s));
            run_dst += run_len;
            run = src;
            run_len = cnt;
        }
        ctx->stats.h2d_bytes += (size_t)npts * sizeof(esfm_dmatch_t) + (size_t)np * (8 + sizeof(PairDesc) + 8) + Kc.size() * 8;
        const int kpp = job.k_per_frame;
        tv_gather_kernel<<<np, 128, 0, s>>>(d_rec.as<esfm_dmatch_t>(), d_frames.as<PairDesc>(), d_kp_off.as<long long>(), d_kp.as<float>(), d_K.as<double>(), kpp,
                                            d_off.as<long long>(), d_n1.as<double2>(), d_n2.as<double2>(), d_bad.as<int>());
        tv_init_kernel<<<(np + 127) / 128, 128, 0, s>>>(d_state.as<TvState>(), d_off.as<long long>(), np, job.params.max_iters, skip_at_most);
        for (int rd = 0; rd < rounds; ++rd) {
            tv_solve_kernel<<<np, kTvRound, 0, s>>>(d_n1.as<double2>(), d_n2.as<double2>(), d_off.as<long long>(), d_state.as<TvState>(), rd,
                                                    (unsigned long long)job.params.seed, 0ull, d_keys.as<unsigned long long>(), d_models.as<double>(), d_nm.as<int>());
            tv_score_kernel<<<dim3(kTvRound / 8, np), 256, 0, s>>>(d_n1.as<double2>(), d_n2.as<double2>(), d_off.as<long long>(), d_K.as<double>(), kpp,
                                                                   job.params.ransac_thre, d_models.as<double>(), d_nm.as<int>(), d_counts.as<int>());
            tv_select_kernel<<<(np + 127) / 128, 128, 0, s>>>(d_state.as<TvState>(), d_off.as<long long>(), np, rd, job.params.ransac_prob, d_models.as<double>(),
                                                              d_nm.as<int>(), d_counts.as<int>());
        }
        tv_pose_kernel<<<np, kTvPoseThreads, 0, s>>>(d_n1.as<double2>(), d_n2.as<double2>(), d_off.as<long long>(), d_K.as<double>(), kpp,
                                                     job.params.ransac_thre, job.params.cheirality_dist, job.params.random_rate, d_state.as<TvState>(),
                                                     d_mask.as<unsigned char>(), d_out.as<esfm_two_view_t>());
        tv_scan_kernel<<<1, kTvScanThreads, 0, s>>>(d_out.as<esfm_two_view_t>(), np, d_inl_off.as<long long>());
        tv_compact_kernel<<<np, kTvPoseThreads, 0, s>>>(d_rec.as<esfm_dmatch_t>(), d_off.as<long long>(), d_mask.as<unsigned char>(), d_inl_off.as<long long>(),
                                                        d_inl.as<esfm_dmatch_t>());
        ctx->stats.kernel_launches += 5 + 3 * (uint64_t)rounds;
        CUDA_TRY(cudaGetLastError());
        int bad = no_bad;
        inl_off.resize((size_t)np + 1);
        CUDA_TRY(cudaMemcpyAsync(&bad, d_bad.p, 4, cudaMemcpyDeviceToHost, s));
        CUDA_TRY(cudaMemcpyAsync(inl_off.data(), d_inl_off.p, (size_t)(np + 1) * 8, cudaMemcpyDeviceToHost, s));
        CUDA_TRY(cudaMemcpyAsync(sh.tv.data() + c0, d_out.p, (size_t)np * sizeof(esfm_two_view_t), cudaMemcpyDeviceToHost, s));
        CUDA_TRY(cudaStreamSynchronize(s));
        if (bad != no_bad) {
            const size_t g = (size_t)sh.ids[(size_t)(c0 + bad)];
            sh.bad_pair = (int64_t)g;
            return fail(ESFM_ERR_INVALID, "pair %zu = (%d,%d): a match's queryIdx or trainIdx is outside its frame's key points", g, r->pairs[g].q_frame, r->pairs[g].t_frame);
        }
        const int64_t total = inl_off[(size_t)np];
        esfm_results::Segment sg{heap_segment_alloc((size_t)total), (size_t)total, nullptr};
        if (!sg.ptr) return fail(ESFM_ERR_NOMEM, "host memory for %lld inlier records", (long long)total);
        sh.segments.push_back(sg);
        if (total > 0) {
            CUDA_TRY(cudaMemcpyAsync(sg.ptr, d_inl.p, (size_t)total * sizeof(esfm_dmatch_t), cudaMemcpyDeviceToHost, s));
            CUDA_TRY(cudaStreamSynchronize(s));
        }
        ctx->stats.d2h_bytes += (size_t)total * sizeof(esfm_dmatch_t) + (size_t)np * sizeof(esfm_two_view_t) + (size_t)(np + 1) * 8 + 4;
        const uint64_t seg = (uint64_t)(sh.segments.size() - 1) << 40;
        for (int p = 0; p < np; ++p) {
            sh.counts[(size_t)(c0 + p)] = sh.tv[(size_t)(c0 + p)].n_inliers;
            sh.offsets[(size_t)(c0 + p)] = seg | (uint64_t)inl_off[(size_t)p];
        }
    }
    return ESFM_OK;
}

int esfm::two_view_assemble(const TvJob& job, std::vector<TvShare>& shares, esfm_results_t** inliers, esfm_two_view_t* out) {
    const esfm_results* r = job.matches;
    esfm_results* res = new (std::nothrow) esfm_results();
    if (!res) return fail(ESFM_ERR_NOMEM, "out of host memory");
    res->kind = r->kind;
    res->ratio = r->ratio;
    res->cross_check = r->cross_check;
    res->frame_rows = r->frame_rows;
    res->pairs = r->pairs;
    res->counts.assign(r->pairs.size(), 0);
    res->offsets.assign(r->pairs.size(), 0);
    for (TvShare& sh : shares) {
        const uint64_t seg_base = (uint64_t)res->segments.size();
        for (auto& sg : sh.segments) res->segments.push_back(sg);
        sh.segments.clear();                       // ownership moved
        for (size_t i = 0; i < sh.ids.size(); ++i) {
            const size_t g = (size_t)sh.ids[i];
            res->counts[g] = sh.counts[i];
            res->offsets[g] = (((sh.offsets[i] >> 40) + seg_base) << 40) | (sh.offsets[i] & kSegOffMask);
            res->total_matches += sh.counts[i];
            out[g] = sh.tv[i];
        }
    }
    *inliers = res;
    return ESFM_OK;
}

extern "C" int esfm_two_view_results(esfm_ctx_t* ctx, esfm_results_t* matches, int n_frames, const int64_t* kp_off, const float* kp_xy, const double* K,
                                     int k_per_frame, const esfm_two_view_params_t* params, int min_pair_matches, esfm_results_t** inliers,
                                     esfm_two_view_t* out) {
    TvJob job;
    if (int rc = two_view_job("esfm_two_view_results", matches, n_frames, kp_off, kp_xy, K, k_per_frame, params, min_pair_matches, inliers, out, &job)) return rc;
    if (!ctx) return fail(ESFM_ERR_INVALID, "esfm_two_view_results: NULL argument");
    std::vector<TvShare> shares(1);
    shares[0].ids.resize(matches->pairs.size());
    for (size_t k = 0; k < shares[0].ids.size(); ++k) shares[0].ids[k] = (int64_t)k;
    if (int rc = two_view_share(ctx, job, shares[0])) return rc;
    return two_view_assemble(job, shares, inliers, out);
}
