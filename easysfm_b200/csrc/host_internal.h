// host_internal.h -- host-side objects behind the opaque handles of include/esfm_match.h, shared by capi.cu (one device)
// and multi.cu (several devices driven by one host process).  Host logic only; every distance / selection / ratio /
// cross-check / compaction step runs in the CUDA kernels of this library.
#pragma once
#include <condition_variable>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <functional>
#include <mutex>
#include <string>
#include <thread>
#include <unordered_map>
#include <vector>

#include "tc_layout.cuh"

namespace esfm {

// ---- error plumbing: one message per host thread (esfm_last_error) -------------------------------------------------
extern thread_local std::string g_last_error;
int fail(int code, const char* fmt, ...);
int set_device(struct ::esfm_ctx* ctx);

#define CUDA_TRY(expr)                                                                                          \
    do {                                                                                                        \
        cudaError_t e__ = (expr);                                                                               \
        if (e__ != cudaSuccess)                                                                                 \
            return ::esfm::fail(ESFM_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__); \
    } while (0)

// A few persistent helper threads that split one large host memcpy (the staging copy of esfm_bank_set_frame: a single core
// copies ~10 GB/s, a 2 MB SURF frame every 0.2 ms; four cores keep up with the PCIe link).
class CopyPool {
public:
    explicit CopyPool(int helpers);
    ~CopyPool();
    void copy(void* dst, const void* src, size_t bytes);   // returns when all of it is copied
private:
    void worker(int k);
    struct Job { char* dst; const char* src; size_t bytes; };
    std::vector<std::thread> threads_;
    std::vector<Job> jobs_;
    std::mutex mu_;
    std::condition_variable cv_work_, cv_done_;
    uint64_t epoch_ = 0;
    int pending_ = 0;
    bool stop_ = false;
};

// Everything one chunk of pairs needs besides the key scratch: two of these let chunk k's matches travel to the host while
// chunk k + 1 is being swept.
struct ChunkBuf {
    PairDesc* d_pairs = nullptr;
    unsigned long long* d_pair_off = nullptr;
    int32_t* d_pair_cnt = nullptr;
    size_t pairs_cap = 0;
    unsigned long long* d_cursor = nullptr;      // [0] arena cursor, [1] overflow flag, [2] rows re-swept by the SURF fallback sweep,
                                                 // [3] train rows put on the verification sweep's gather lists
    esfm_dmatch_t* arena = nullptr;              // dense match arena of the chunk
    size_t arena_cap = 0;                        // in matches
    uint64_t generation = 0;                     // bumped whenever the arena is overwritten
    // pinned host memory
    PairDesc* h_pairs = nullptr;   size_t h_pairs_cap = 0;     // launch-ordered pair list (upload)
    unsigned char* h_meta = nullptr; size_t h_meta_bytes = 0;  // cursor + offsets + counts (download)
    cudaEvent_t ev_t0 = nullptr, ev_t1 = nullptr, ev_t2 = nullptr;   // sweep start / sweep end / finalize end
    cudaEvent_t ev_v0 = nullptr, ev_v1 = nullptr;                    // two-phase cross-check: verification sweep start / end
    bool two_phase = false;                      // the chunk last run here had a verification sweep (ev_v0 / ev_v1 are valid)
    cudaEvent_t ev_meta = nullptr, ev_copied = nullptr;
    bool copy_pending = false;                   // a device->host copy of the arena may still be in flight (ev_copied)
};

struct OrbState;                                 // scratch of the ORB extractor (orb.cu), kept between calls

// The tensor-core operand image of a bank (tc_layout.cuh), built for the sweep that reads it.  SURF: the 3xTF32 hi / lo split (sweep_l2_tc.cu)
// or the 16-bit "H" split (sweep_win.cu; followed by what win_fast_eps needs).  ORB: FP8 +-1 (sweep_l2_tc.cu's generic epilogue,
// sweep_win.cu) or the FP8 "Z" encoding, whose accumulator is the packed key (sweep_l2_tc.cu).
enum class TcImage { Tf32x3, H, Fp8Pm1, Fp8Z };

}  // namespace esfm

struct esfm_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    cudaStream_t copy_stream = nullptr;    // device->host traffic of finished chunks
    cudaMemPool_t mempool = nullptr;       // private stream-ordered pool for banks: freed blocks stay cached, and die with the ctx
    int sm_count = 0;
    bool profiling = true;
    int orb_z = 1;                         // ORB tensor-core sweep with the "Z" operand encoding (packed keys from the MMA): default;
                                           // $ESFM_ORB_Z=0 selects the +-1 encoding with the generic epilogue
    int hamming_engine = ESFM_HAMMING_ENGINE_TC16;
    int l2_engine = ESFM_L2_ENGINE_TC16;
    esfm_stats_t stats{};
    // device scratch, grown on demand
    esfm::u64* keys = nullptr;     size_t keys_bytes = 0;
    uint32_t* col_thr = nullptr;   size_t col_thr_elems = 0;
    int* gather_cnt = nullptr;     size_t gather_cnt_elems = 0;     // two-phase cross-check: train rows to verify, per pair of the chunk
    int tc16_exact = 0;                    // $ESFM_TC16_EXACT=1: SURF tc16 sweeps in exact mode (13 MMA slots per tile) instead of fast mode
                                           // (9 slots) + exact fallback sweep of the rows it cannot settle
    esfm::ChunkBuf buf[2];
    // a pool of large pinned buffers that banks (upload staging) and results (downloaded matches) borrow, so steady-state
    // calls never allocate or zero-fill host memory
    struct Pinned { void* ptr; size_t bytes; bool in_use; };
    std::vector<Pinned> pool;
    esfm::CopyPool* copier = nullptr;
    // Matches of a multi-chunk batch reach pageable host memory through a FEW SMALL pinned slots, piece by piece (device->host
    // copy of piece i + 1 overlapped with the host copy of piece i): allocating pinned memory costs ~1 s per GB, so whole-chunk
    // pinned buffers would cost more than the sweeps of a job that runs a handful of chunks per device.
    static constexpr int kSlots = 4;
    static constexpr size_t kSlotMatches = (size_t)2 << 20;     // 2 Mi matches = 32 MB per slot
    esfm_dmatch_t* h_slot[kSlots] = {nullptr, nullptr, nullptr, nullptr};
    cudaEvent_t ev_slot[kSlots] = {nullptr, nullptr, nullptr, nullptr};
    esfm_dmatch_t* h_scratch = nullptr; size_t h_scratch_cap = 0;   // pageable scratch of digests-only batches (one chunk's matches)
    esfm::OrbState* orb = nullptr;
    struct esfm_bank* pair_bank[2] = {nullptr, nullptr};   // reusable two-frame banks of esfm_match_descriptors, one per kind
};

struct esfm_bank {
    esfm_ctx* ctx = nullptr;
    int kind = 0;
    int n_frames = 0;
    std::vector<int> rows;                    // per frame, -1 = not set
    // upload staging: frames are appended to a pinned host buffer and copied to its device mirror right away, so the
    // host->device traffic of frame k overlaps the staging copy of frame k + 1; frames set in order make the mirror the bank
    uint8_t* h_up = nullptr;
    uint8_t* d_up = nullptr;
    size_t up_cap = 0, up_used = 0;
    std::vector<size_t> host_off;             // per frame offset into the staging buffers ((size_t)-1 = no host data)
    std::vector<const void*> host_ext;        // per frame caller-owned pinned source (esfm_bank_set_frame_pinned), else nullptr
    bool committed = false;
    bool device_allocated = false;
    // device
    void* d_rows = nullptr;  size_t rows_bytes = 0;  size_t rows_cap = 0;
    float* d_kmajor = nullptr; size_t kmajor_bytes = 0; size_t kmajor_cap = 0;   // FFMA engine operand tiles, built on its first sweep
    bool kmajor_built = false;
    unsigned char* d_tc = nullptr; size_t tc_bytes = 0; size_t tc_cap = 0;       // tensor-core operand images, built on first use
    bool tc_built = false;
    esfm::TcImage tc_image = esfm::TcImage::Tf32x3;       // ... which one
    int* d_tables = nullptr;                              // frame_rows | row_off | tile_off, (n_frames + 1) ints each
    int* d_frame_rows = nullptr;
    int* d_row_off = nullptr;
    int* d_tile_off = nullptr;
    // host copies
    std::vector<int> row_off, tile_off;
    int max_rows = 0;
    // F32X64, measured at commit: the largest |x| of any component, and the smallest of the non-empty frames' largest |x| (plan_sweep routes
    // on both)
    float abs_max = 0.f, frame_abs_min = 0.f;
    size_t row_bytes() const { return kind == ESFM_KIND_F32X64 ? esfm::kDim * sizeof(float) : 32; }
};

struct esfm_results {
    esfm_ctx* ctx = nullptr;
    std::vector<esfm::PairDesc> pairs;
    std::vector<int32_t> counts;
    std::vector<uint64_t> offsets;          // segment index << 40 | offset (in matches) inside that segment
    struct Segment {
        esfm_dmatch_t* ptr; size_t count;
        esfm_ctx* pool_ctx;                 // pinned buffer borrowed from this context's pool; nullptr = plain heap memory
    };
    std::vector<Segment> segments;
    std::vector<uint64_t> digests;          // per-pair digest of the matches (ESFM_KEEP_DIGESTS, or computed on demand)
    int keep = ESFM_KEEP_MATCHES;
    int kind = -1, cross_check = 0;         // what the batch was matched with (kept in the match file)
    double ratio = 0.0;
    std::vector<int32_t> frame_rows;        // rows of every frame of the bank it was matched on (empty: unknown, a version-1 file)
    std::unordered_map<uint64_t, int64_t> index;
    bool fetched = true;
    // device-resident variant (single chunk only)
    int dev_buf = 0;
    uint64_t arena_generation = 0;
    uint64_t device_matches = 0;
    int64_t total_matches = 0;
};

namespace esfm {

struct MatchOpts {
    bool fetch = true;               // copy the matches to the host
    int keep = ESFM_KEEP_MATCHES;    // ... and keep them, or only their per-pair digests
};

int match_pairs_impl(esfm_bank* b, const esfm_pair_t* pairs, int64_t n_pairs, double ratio, int cross_check, const MatchOpts& opts,
                     esfm_results** out);
uint64_t digest_matches(const esfm_dmatch_t* m, int n);
void* pool_acquire(esfm_ctx* ctx, size_t bytes, size_t* got);
void pool_release(esfm_ctx* ctx, void* ptr);
esfm_dmatch_t* heap_segment_alloc(size_t n_matches);
// orb.cu: the extractor behind esfm_orb_extract / esfm_bank_set_frame_from_image.  `sink`, when set, is called once the number of key points
// is known and returns the device address the n x 32 descriptor bytes go to (nullptr: the extractor's own scratch).
using OrbSink = std::function<int(int n, uint8_t** d_dst)>;
int orb_extract_impl(esfm_ctx* ctx, const unsigned char* image, int rows, int cols, int channels, size_t row_stride, int max_features,
                     esfm_keypoint_t* keypoints, unsigned char* h_desc, int capacity, int* n_out, const OrbSink& sink);
void orb_state_destroy(esfm_ctx* ctx);
int reserve_stream_slots(esfm_ctx* ctx);     // allocate the pinned slots now (esfm_multi_init: outside any job's clock)

// two_view.cu: verification of a results batch (esfm_two_view_results, esfm_multi_two_view_results).  The arguments of one call, checked once
// by two_view_job, and what one device makes of its share of the batch's pairs.
struct TvJob {
    const esfm_results* matches = nullptr;
    int n_frames = 0;
    const int64_t* kp_off = nullptr;
    const float* kp_xy = nullptr;
    const double* K = nullptr;
    int k_per_frame = 0;
    esfm_two_view_params_t params{};
    int min_pair_matches = 0;
};
struct TvShare {
    std::vector<int64_t> ids;                        // batch positions of the share's pairs, ascending
    std::vector<int32_t> counts;                     // inliers per pair
    std::vector<uint64_t> offsets;                   // segment index << 40 | offset of the pair's inliers in `segments`
    std::vector<esfm_results::Segment> segments;     // heap memory, one per chunk
    std::vector<esfm_two_view_t> tv;
    int64_t bad_pair = -1;                           // batch position of the first pair with a match index outside its frame's key points
    TvShare() = default;
    TvShare(const TvShare&) = delete;
    TvShare& operator=(const TvShare&) = delete;
    ~TvShare() { for (auto& s : segments) free(s.ptr); }
};
int two_view_job(const char* who, esfm_results* matches, int n_frames, const int64_t* kp_off, const float* kp_xy, const double* K, int k_per_frame,
                 const esfm_two_view_params_t* params, int min_pair_matches, esfm_results_t** inliers, esfm_two_view_t* out, TvJob* job);
int two_view_share(esfm_ctx* ctx, const TvJob& job, TvShare& share);
// One results batch in the caller's pair order from the shares (their segments are adopted), and every pair's record to out.
int two_view_assemble(const TvJob& job, std::vector<TvShare>& shares, esfm_results_t** inliers, esfm_two_view_t* out);

}  // namespace esfm
