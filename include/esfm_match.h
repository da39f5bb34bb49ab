/*
 * esfm_match.h -- C ABI of libesfm_match.so: B200-native (sm_100a) all-pairs descriptor matching,
 * the drop-in for EasySFM's matching hot path.  Plain pointers and sizes only; no C++/torch types.
 *
 * Every entry point names the reference interface it replaces (paths relative to the EasySFM tree):
 *   - p3dv::FeatureMatching::matchFeaturesORB   cpp_code/include/feature_matching.h:17-18,
 *                                               cpp_code/src/feature_matching.cpp:71-113
 *   - p3dv::FeatureMatching::matchFeaturesSURF  cpp_code/include/feature_matching.h:20-21,
 *                                               cpp_code/src/feature_matching.cpp:115-158
 *   - the all-pairs driver loop                 cpp_code/test/sfm.cpp:140-161  (query = frame i, train = frame j < i)
 *   - frame_t::descriptors / frame_pair_t::matches   cpp_code/include/utility.h:31,62
 *   - Python pairwise_match matcher calls       python_code/feature_match.py:24-39
 *
 * Semantics (identical to OpenCV BFMatcher as the reference calls it; see DESIGN.md):
 *   forward brute-force 2-NN (L2 on 64 x fp32, Hamming on 256 bits), lowest train index on ties;
 *   keep NN1 iff (double)d1 < ratio * (double)d2  (feature_matching.cpp:88,133);
 *   if cross_check: keep (q,t) only if q is the nearest query row of train row t (lowest index on ties)
 *   (feature_match.py:26-27); output in ascending queryIdx with imgIdx = 0 (feature_matching.cpp:84-91).
 *   A train frame with fewer than 2 rows yields zero matches (the reference reads out of bounds there).
 *   ratio = +infinity disables the ratio test (no second neighbour needed): with cross_check = 1 that is
 *   cv2.BFMatcher(norm, crossCheck=True).match of feature_match.py:26-27, in ascending queryIdx.
 *   cross_check = 0 with ESFM_KIND_B256 reproduces matchFeaturesORB exactly.
 *
 * Error convention: every function returns 0 on success and a nonzero esfm_status otherwise; nothing
 * throws across the boundary; esfm_last_error() returns a message for the calling thread's last failure.
 * There is NO CPU fallback: without a CUDA device every compute entry point fails with ESFM_ERR_CUDA.
 *
 * Threading: one host thread drives one context; calls on one context are not re-entrant.  esfm_multi_* (several GPUs of one
 * box from ONE host process, the shape of the reference's single-process caller cpp_code/test/sfm.cpp:32) starts one worker
 * thread per device internally; the caller still makes one call.
 */
#ifndef ESFM_MATCH_H_
#define ESFM_MATCH_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ESFM_ABI_VERSION 2

typedef enum esfm_status {
    ESFM_OK = 0,
    ESFM_ERR_INVALID = 1,  /* bad argument (null pointer, wrong cols/kind, index out of range, ...) */
    ESFM_ERR_CUDA = 2,     /* CUDA runtime / driver failure, or no usable device */
    ESFM_ERR_STATE = 3,    /* call order violated (e.g. matching before esfm_bank_commit) */
    ESFM_ERR_NOMEM = 4,    /* host or device allocation failed */
    ESFM_ERR_CAPACITY = 5  /* caller-provided output buffer too small, or frame too large for the kernels */
} esfm_status;

/* Descriptor kinds: the two the reference produces (feature_matching.cpp:16-22 ORB 32 bytes, :45-52 SURF 64 floats). */
typedef enum esfm_kind {
    ESFM_KIND_F32X64 = 0, /* SURF: rows x 64 float32, L2 distance          (cv::Mat CV_32FC1) */
    ESFM_KIND_B256 = 1    /* ORB : rows x 32 uint8 (256 bits), Hamming     (cv::Mat CV_8UC1)  */
} esfm_kind;

/* Layout-identical to cv::DMatch (16 bytes) so a C++ shim can insert() it straight into std::vector<cv::DMatch>. */
typedef struct esfm_dmatch_t {
    int32_t queryIdx;
    int32_t trainIdx;
    int32_t imgIdx; /* always 0, as in the reference */
    float distance; /* L2: sqrt(sum (a-b)^2); Hamming: bit count as float */
} esfm_dmatch_t;

/* One unit of the pair schedule: match frame `query` (rows = queries) against frame `train`. */
typedef struct esfm_pair_t {
    int32_t query;
    int32_t train;
} esfm_pair_t;

typedef struct esfm_ctx esfm_ctx_t;         /* one CUDA device + stream + scratch */
typedef struct esfm_bank esfm_bank_t;       /* device-resident descriptor bank (all frames of one kind) */
typedef struct esfm_results esfm_results_t; /* host-resident compacted matches of a batch of pairs */

/* Counters a caller (bench.py) reads back; all cumulative since esfm_init. */
typedef struct esfm_stats_t {
    uint64_t kernel_launches;  /* CUDA kernels launched by this library */
    uint64_t h2d_bytes;        /* host->device bytes copied */
    uint64_t d2h_bytes;        /* device->host bytes copied */
    uint64_t comparisons;      /* descriptor comparisons evaluated (rows_q * rows_t per pair, counted once) */
    uint64_t pairs;            /* image pairs matched */
    double last_sweep_ms;      /* device time of the most recent distance/top-2 sweep kernel (CUDA events; SURF tc16: with the fallback sweep) */
    double last_finalize_ms;   /* device time of the most recent refine/ratio/cross-check/compaction kernel */
    double sweep_ms_total;     /* sum of sweep kernel device times */
    uint64_t sweep_launches;   /* number of sweep kernel launches */
    uint64_t fallback_rows;    /* SURF tc16: query rows the 9-slot sweep could not settle, re-swept in exact (13-slot) mode */
    uint64_t verified_rows;    /* tc16 cross-check: train rows the ratio-test histograms could not decide, re-swept by the verification sweep */
} esfm_stats_t;

int esfm_abi_version(void);

/* Message for the calling thread's most recent failing call ("" if none). Never NULL. */
const char* esfm_last_error(void);

/* ---- context ------------------------------------------------------------------------------- */

/* Bind a context to CUDA device `device`.  `cuda_stream` is a cudaStream_t to launch on (so the caller
 * can bracket work with its own CUDA events), or NULL to let the library create its own stream. */
int esfm_init(int device, void* cuda_stream, esfm_ctx_t** ctx);
int esfm_destroy(esfm_ctx_t* ctx);
int esfm_synchronize(esfm_ctx_t* ctx);
int esfm_get_stats(esfm_ctx_t* ctx, esfm_stats_t* out);
/* Time the sweep/finalize kernels with CUDA events (default on; costs two event records per launch). */
int esfm_set_profiling(esfm_ctx_t* ctx, int enabled);
/* Number of SMs of the bound device (grid sizing is a multiple of this). */
int esfm_device_sm_count(esfm_ctx_t* ctx, int* sms);

/* Which kernel serves ESFM_KIND_F32X64 sweeps.  Both produce the same candidates for finalize's direct-form
 * re-evaluation (the reference's arithmetic, BFMatcher(NORM_L2): feature_match.py:33-34); they differ in how the
 * RANKING distance is computed:
 *   ESFM_L2_ENGINE_FFMA  exact-FP32 FFMA expansion  1/2|q|^2 + 1/2|t|^2 - q.t  on the FP32 pipe;
 *   ESFM_L2_ENGINE_TC    the same quantity as a 3xTF32 split product on the tcgen05 tensor cores;
 *   ESFM_L2_ENGINE_TC16  the same quantity as a two-term FP16 split product (kind::f16, fp32 accumulation: the error of 3xTF32 at
 *                        half the tensor-pipe time and half the operand bytes), rows reported as (value, slice of columns) and
 *                        resolved exactly by the finalize pass.
 * Default: $ESFM_L2_ENGINE ("ffma" | "tc" | "tc16") at esfm_init, else ESFM_L2_ENGINE_TC16. */
#define ESFM_L2_ENGINE_FFMA 0
#define ESFM_L2_ENGINE_TC 1
#define ESFM_L2_ENGINE_TC16 2
int esfm_set_l2_engine(esfm_ctx_t* ctx, int engine);
int esfm_get_l2_engine(esfm_ctx_t* ctx, int* engine);
/* Which kernel serves ESFM_KIND_B256: XOR + POPC on the integer pipes (the north-star design), or the same Hamming
 * distance as an exact FP8 dot product on the tcgen05 tensor cores (bits become +-2^k, the fp32 accumulator holds the
 * integer 20480 + 2^15 * hamming + column exactly; 2.3x faster).
 * ESFM_HAMMING_ENGINE_TC16: the FP8 +-1 dot product with FP16 accumulators (-2 * hamming, exact), a selection epilogue on packed
 * halves, rows reported as (distance, slice of 32 columns) and resolved with XOR + POPC by the finalize pass.  All three are
 * bit-exact against OpenCV and against each other;
 * default: $ESFM_HAMMING_ENGINE ("popc" | "tc" | "tc16") at esfm_init, else ESFM_HAMMING_ENGINE_TC16. */
#define ESFM_HAMMING_ENGINE_POPC 0
#define ESFM_HAMMING_ENGINE_TC 1
#define ESFM_HAMMING_ENGINE_TC16 2
int esfm_set_hamming_engine(esfm_ctx_t* ctx, int engine);
int esfm_get_hamming_engine(esfm_ctx_t* ctx, int* engine);

/* ---- descriptor bank (replaces the per-call cv::Mat arguments; utility.h:31) ---------------- */

int esfm_bank_create(esfm_ctx_t* ctx, esfm_kind kind, int n_frames, esfm_bank_t** bank);
/* Copy one frame's descriptors (frame_t::descriptors: .data, .rows, .cols, .step).  cols must be 64
 * (F32X64, elements are float) or 32 (B256, elements are uint8).  rows may be 0.  The host pointer
 * need not outlive the call.  `frame_id` in [0, n_frames).  May be called again before commit. */
int esfm_bank_set_frame(esfm_bank_t* bank, int frame_id, const void* data, int rows, int cols, size_t step_bytes);
/* Same, without the host-side copy: `data` must be page-locked (cudaMallocHost / cudaHostRegister) with
 * step_bytes == the row size, and must stay valid and unmodified until esfm_bank_commit returns; commit copies
 * straight from it (one async host->device copy per frame).  For callers that already hold their descriptors in
 * pinned memory (a feature extractor writing into a pinned arena); cv::Mat data is pageable: use esfm_bank_set_frame.
 * ESFM_ERR_INVALID if the memory is not page-locked or the rows are not densely packed. */
int esfm_bank_set_frame_pinned(esfm_bank_t* bank, int frame_id, const void* data, int rows, int cols, size_t step_bytes);
/* Declare a frame's row count without host data: for banks whose rows arrive on the device
 * (esfm_bank_device_rows + an NCCL broadcast driven by the host process, see INTEGRATION.md). */
int esfm_bank_set_frame_rows(esfm_bank_t* bank, int frame_id, int rows);
/* Pack -> one host->device copy -> derived device layouts (k-major tiles + half squared norms for
 * F32X64).  After commit the bank is immutable and resident in HBM until destroyed. */
int esfm_bank_commit(esfm_bank_t* bank);
/* Allocate device storage from the declared row counts only (no host data, no copy). */
int esfm_bank_alloc_device(esfm_bank_t* bank);
/* Raw row-major device buffer of all frames back to back (frame f starts at row offset sum(rows[<f])):
 * F32X64 -> float[total_rows][64], B256 -> uint8[total_rows][32].  Valid after commit/alloc_device. */
int esfm_bank_device_rows(esfm_bank_t* bank, void** dev_ptr, size_t* bytes);
/* Rebuild the derived layouts after the caller wrote the raw device buffer (e.g. by broadcast). */
int esfm_bank_commit_device(esfm_bank_t* bank);
int esfm_bank_n_frames(esfm_bank_t* bank, int* n_frames);
int esfm_bank_frame_rows(esfm_bank_t* bank, int frame_id, int* rows);
int esfm_bank_device_bytes(esfm_bank_t* bank, size_t* bytes);
int esfm_bank_destroy(esfm_bank_t* bank);

/* ---- matching ------------------------------------------------------------------------------ */

/* All N(N-1)/2 pairs of the bank in the reference's loop order: for i in [0,N): for j in [0,i):
 * query = i, train = j  (sfm.cpp:140-161). */
int esfm_match_all_pairs(esfm_bank_t* bank, double ratio, int cross_check, esfm_results_t** results);
/* An explicit batch of pairs (the unit a multi-GPU scheduler shards). */
int esfm_match_pairs(esfm_bank_t* bank, const esfm_pair_t* pairs, int64_t n_pairs, double ratio, int cross_check,
                     esfm_results_t** results);
/* Same, but matches stay on the device (no device->host copy); only counts are returned to the host.
 * Used to measure the device-resident throughput; results can still be fetched with esfm_results_fetch. */
int esfm_match_pairs_device(esfm_bank_t* bank, const esfm_pair_t* pairs, int64_t n_pairs, double ratio,
                            int cross_check, esfm_results_t** results);
int esfm_results_fetch(esfm_results_t* results);
/* Largest batch of pairs of this bank that the library processes as ONE chunk (bounded scratch: <= 4 GB of keys, <= 2 GB of
 * match arena, <= 65536 pairs); only a one-chunk device-resident batch can be fetched / read on the device afterwards. */
int esfm_bank_chunk_pairs(esfm_bank_t* bank, int64_t* max_pairs);
/* One pair, caller-owned output (the unmodified per-call shape of matchFeaturesORB/SURF).
 * `cap` = capacity of `out` in matches (rows of the query frame is always enough). */
int esfm_match_pair(esfm_bank_t* bank, int query_frame, int train_frame, double ratio, int cross_check,
                    esfm_dmatch_t* out, int cap, int* n_matches);
/* Two host descriptor matrices in, matches out: literally the reference's call
 * matchFeaturesX(frame_1 = query, frame_2 = train, matches, ratio).  Uploads both, matches, frees. */
int esfm_match_descriptors(esfm_ctx_t* ctx, esfm_kind kind, const void* query, int rows_q, size_t step_q,
                           const void* train, int rows_t, size_t step_t, int cols, double ratio, int cross_check,
                           esfm_dmatch_t* out, int cap, int* n_matches);
/* Raw 2-NN of one pair (knnMatch(k=2), feature_matching.cpp:80): idx[2*q+r], dist[2*q+r], r in {0,1};
 * idx = -1 / dist = +inf where the train frame has fewer rows. */
int esfm_knn2_pair(esfm_bank_t* bank, int query_frame, int train_frame, int32_t* idx, float* dist);

/* What a batch keeps on the host.  The whole-job configs produce more matches than a host should hold at once
 * (5000 images x 4k ORB features: ~2e10 match records), so a batch can keep only a 64-bit digest per pair (count, indices and
 * distance bits of its matches folded in order) -- enough to compare runs across GPU counts -- next to the per-pair counts. */
#define ESFM_KEEP_MATCHES 0
#define ESFM_KEEP_DIGESTS 1
/* esfm_match_pairs with an explicit keep mode (ESFM_KEEP_DIGESTS: matches are downloaded chunk by chunk, digested, dropped). */
int esfm_match_pairs_keep(esfm_bank_t* bank, const esfm_pair_t* pairs, int64_t n_pairs, double ratio, int cross_check, int keep,
                          esfm_results_t** results);

/* ---- results (replaces frame_pair_t::matches, utility.h:62) -------------------------------- */

int esfm_results_counts(esfm_results_t* results, int64_t* n_pairs, int64_t* n_matches);
/* k-th pair of the batch in submission order. */
int esfm_results_pair_at(esfm_results_t* results, int64_t k, int* query_frame, int* train_frame,
                         const esfm_dmatch_t** matches, int* n_matches);
/* Lookup by frame ids (first occurrence in the batch). */
int esfm_results_pair(esfm_results_t* results, int query_frame, int train_frame, const esfm_dmatch_t** matches,
                      int* n_matches);
/* Per-pair match counts for the whole batch (n_pairs int32 values). */
int esfm_results_pair_counts(esfm_results_t* results, int32_t* counts);
/* Bulk accessor: every pair's matches back to back in batch order, in ONE call (n_matches records, esfm_results_counts);
 * `offsets` (optional, n_pairs + 1 entries) receives where each pair starts.  ESFM_ERR_CAPACITY if `cap` is too small. */
int esfm_results_copy_all(esfm_results_t* results, esfm_dmatch_t* out, int64_t cap, int64_t* offsets);
/* Zero-copy view of a fetched batch: its matches live in a few host segments (one per chunk and device); every pair's matches
 * are contiguous inside one of them.  esfm_results_pair_layout fills, per pair, the segment index and the offset (in matches)
 * inside it; esfm_results_segment_at returns a segment.  Valid until esfm_results_destroy. */
int esfm_results_segment_count(esfm_results_t* results, int* n_segments);
int esfm_results_segment_at(esfm_results_t* results, int segment, const esfm_dmatch_t** matches, int64_t* n_matches);
int esfm_results_pair_layout(esfm_results_t* results, int32_t* segment, int64_t* offset);
/* Per-pair 64-bit digests (n_pairs values): stored ones for ESFM_KEEP_DIGESTS batches, else computed from the matches. */
int esfm_results_digests(esfm_results_t* results, uint64_t* digests);
/* Device-resident batch (esfm_match_pairs_device, one chunk): the dense match arena on the device, pairs back to back in LAUNCH
 * order (`device_offsets` of esfm_results_device_layout); valid until the next matching call on the context.  For callers that
 * move matches between GPUs themselves (the one-process-per-GPU scheduler: NCCL send of this buffer). */
int esfm_results_device_matches(esfm_results_t* results, void** dev_ptr, int64_t* n_matches);
/* Offset (in matches) of every pair of a device-resident batch inside that arena (n_pairs values). */
int esfm_results_device_layout(esfm_results_t* results, int64_t* offsets);
int esfm_results_destroy(esfm_results_t* results);

/* ---- persistence (SURVEY 8f rank 2: restart the SfM pipeline after matching) --------------------
 * The reference keeps every pair's matches in RAM only (img_match_graph, sfm.cpp:130-197) and re-matches on
 * every run.  esfm_results_save writes a fetched batch to one little-endian file:
 *   "ESFMMTCH" | u32 version = 1 | u32 sizeof(esfm_dmatch_t) = 16 | i64 n_pairs | i64 n_matches |
 *   i32 kind | i32 cross_check | f64 ratio |
 *   n_pairs x esfm_pair_t {query, train} | n_pairs x i32 counts | n_matches x esfm_dmatch_t (pairs in batch order)
 * esfm_results_load needs no device and no context: the loaded batch answers esfm_results_counts / _pair_at /
 * _pair / _pair_counts exactly like the one that was saved.  ESFM_ERR_INVALID on a missing, truncated or
 * foreign file. */
int esfm_results_save(esfm_results_t* results, const char* path);
/* The parameters the batch was matched with (also stored in the file, so a resumed run can check them). */
int esfm_results_params(esfm_results_t* results, int* kind, double* ratio, int* cross_check);
int esfm_results_load(const char* path, esfm_results_t** results);
/* Row counts of the frames the batch was matched on (n_frames = 0: unknown, a version-1 file); rows may be NULL. */
int esfm_results_frame_rows(esfm_results_t* results, int32_t* rows, int cap, int* n_frames);
/* ESFM_OK iff the batch fits a frame list with these row counts: stored row counts equal, every pair inside [0, n_frames),
 * every match index inside its frames' rows.  Call it after esfm_results_load before trusting the indices. */
int esfm_results_validate(esfm_results_t* results, int n_frames, const int32_t* rows);

/* ---- track building and co-visibility (SURVEY 8f rank 3: what consumes the matches next) ---------------------------------
 * cpp_code/test/sfm.cpp:140-217: every keypoint gets a unique point id; the inlier matches of pair (i, j) label frame i's
 * keypoints with frame j's ids unless that id is already used in frame i; unlabelled keypoints get fresh ids after the row.
 * The labelling is order-dependent, so pairs must be fed in the reference's loop order (i ascending, j < i ascending).
 * cpp_code/src/feature_matching.cpp:160-233 (findInitializeFramePair) then scores EVERY frame pair by the points both see,
 * weighted by how many frames see each point -- O(N^2 P) on a dense bool matrix in the reference, one CUDA kernel over sorted
 * id lists here -- and :235-268 (findNextFrame) picks the frame that sees most of the current 3D points.
 * Integer work: results are identical to the reference's loops (oracle/tracks_oracle.c, tests/test_tracks.py). */
typedef struct esfm_tracks esfm_tracks_t;
int esfm_tracks_create(int n_frames, const int32_t* keypoints_per_frame, esfm_tracks_t** tracks);
int esfm_tracks_destroy(esfm_tracks_t* tracks);
/* The inlier matches of pair (frame_i = query, frame_j = train), sfm.cpp:172-194.  frame_i must be the frame in progress. */
int esfm_tracks_add_pair(esfm_tracks_t* tracks, int frame_i, int frame_j, const esfm_dmatch_t* inlier_matches, int n);
/* End of frame_i's row: fresh ids for its unlabelled keypoints, its row of the track matrix (sfm.cpp:199-213). */
int esfm_tracks_finish_frame(esfm_tracks_t* tracks, int frame_i);
/* The whole loop over a batch holding all pairs in loop order: pairs with more than min_pair_matches matches contribute all of them.
 * The reference feeds each pair's RANSAC inliers (sfm.cpp:163-194), so its tracks come from the verified batch of
 * esfm_two_view_results (pairs at or below 20 matches already have no inliers there) with min_pair_matches = 0; a matched batch
 * (esfm_match_all_pairs / esfm_multi_match_all_pairs) with min_pair_matches = 20 gives the tracks of unverified matches. */
int esfm_tracks_build(esfm_tracks_t* tracks, esfm_results_t* results, int min_pair_matches);
/* frame_t::unique_pixel_ids / unique_pixel_has_match of one frame (library-owned, n = its keypoints). */
int esfm_tracks_frame(esfm_tracks_t* tracks, int frame, const int32_t** unique_pixel_ids, const uint8_t** unique_pixel_has_match, int* n);
int esfm_tracks_counts(esfm_tracks_t* tracks, int* frames_done, int64_t* n_unique_points);
/* Co-visibility score of every pair in loop order (n_frames (n_frames - 1) / 2 values), computed on ctx's device;
 * kernel_ms (optional) = device time of the scoring kernel. */
int esfm_tracks_pair_scores(esfm_ctx_t* ctx, esfm_tracks_t* tracks, int64_t* scores, double* kernel_ms);
/* findInitializeFramePair (defaults of feature_matching.h:26-27: min_track_num_init 100, max_depth_baseline_ratio_init 50.0).
 * appro_depth = frame_pair_t::appro_depth per pair in loop order, or NULL (1.0).  *found = 0: no pair qualified, the reference's
 * fallback (1, 0) is returned. */
int esfm_tracks_find_init_pair(esfm_ctx_t* ctx, esfm_tracks_t* tracks, const double* appro_depth, int min_track_num_init,
                               double max_depth_baseline_ratio_init, int* frame_1, int* frame_2, double* depth_init,
                               int64_t* best_score, int* found);
/* findNextFrame: among frames with frames_to_process[f] != 0 the one that sees most of point_ids (first best wins; *next_frame
 * is left untouched when none sees any). */
int esfm_tracks_find_next_frame(esfm_tracks_t* tracks, const uint8_t* frames_to_process, const int32_t* point_ids, int64_t n_ids,
                                int* next_frame, int* common_points);

/* ---- several GPUs of one box, one host process (SURVEY 8b/8e; caller: the single-threaded pair loop sfm.cpp:140-161) -----
 * esfm_multi_init binds n devices (ids = NULL: devices 0..n-1).  A multi bank is fed like a bank (set_frame x N, or through
 * its primary replica on device 0); esfm_multi_bank_commit uploads it to device 0, replicates the raw descriptors on the other
 * devices with ONE ncclBroadcast over NVLink (NCCL is loaded at run time: libnccl.so.2, or $ESFM_NCCL_LIBRARY) and builds
 * the derived layouts on every device.  esfm_multi_match_* deals blocks of consecutive pairs to the devices by work
 * (rows_q * rows_t), runs one worker thread + stream per device, returns each device's matches over its own PCIe link
 * chunk by chunk (the copy of chunk k overlaps the sweep of chunk k + 1) and merges them into ONE results object in the
 * caller's pair order: byte-identical to the single-device result.  No inter-GPU traffic during matching.
 * The same device may be listed several times (tests on a one-GPU box): its replicas are then filled by device copies. */
typedef struct esfm_multi esfm_multi_t;
typedef struct esfm_multi_bank esfm_multi_bank_t;
typedef struct esfm_multi_timing_t {
    double broadcast_ms;      /* last esfm_multi_bank_commit: replication of the raw bank on devices 1..n-1 (host wall clock) */
    double commit_ms;         /* last esfm_multi_bank_commit: the whole call */
    double match_ms;          /* last esfm_multi_match_* or esfm_multi_two_view_results: the whole call (host wall clock, results merged) */
    double device_ms_max;     /* ... slowest device's share */
    double device_ms_min;     /* ... fastest device's share */
    double work_imbalance;    /* max over devices of assigned comparisons (verification: matches) / mean, minus 1 */
    int used_nccl;            /* 1 = ncclBroadcast, 0 = device copies (one device, or a device listed twice) */
} esfm_multi_timing_t;

int esfm_multi_init(int n_devices, const int* device_ids, esfm_multi_t** multi);
int esfm_multi_destroy(esfm_multi_t* multi);
int esfm_multi_device_count(esfm_multi_t* multi, int* n_devices);
/* Borrowed per-device context (engine selection, stats); k in [0, n_devices). */
int esfm_multi_ctx(esfm_multi_t* multi, int k, esfm_ctx_t** ctx);
int esfm_multi_timing(esfm_multi_t* multi, esfm_multi_timing_t* out);

int esfm_multi_bank_create(esfm_multi_t* multi, esfm_kind kind, int n_frames, esfm_multi_bank_t** bank);
int esfm_multi_bank_set_frame(esfm_multi_bank_t* bank, int frame_id, const void* data, int rows, int cols, size_t step_bytes);
/* Borrowed device-0 replica, for every other way of filling a bank (esfm_bank_set_frame_pinned, or esfm_bank_set_frame_rows +
 * esfm_bank_alloc_device + esfm_bank_device_rows when the descriptors are produced on the device).  Do not commit it. */
int esfm_multi_bank_primary(esfm_multi_bank_t* bank, esfm_bank_t** primary);
int esfm_multi_bank_commit(esfm_multi_bank_t* bank);
int esfm_multi_bank_destroy(esfm_multi_bank_t* bank);
/* All N(N-1)/2 pairs in the reference's loop order (sfm.cpp:140-161), or an explicit list; keep = ESFM_KEEP_MATCHES | _DIGESTS. */
int esfm_multi_match_all_pairs(esfm_multi_bank_t* bank, double ratio, int cross_check, int keep, esfm_results_t** results);
int esfm_multi_match_pairs(esfm_multi_bank_t* bank, const esfm_pair_t* pairs, int64_t n_pairs, double ratio, int cross_check,
                           int keep, esfm_results_t** results);

/* ---- SURVEY 8f rank 1: two-view geometric verification of the matches, batched over image pairs ------------------------------------------
 * Replaces MotionEstimator::estimate2D2D_E5P_RANSAC (cpp_code/src/estimate_motion.cpp:27-97; decl cpp_code/include/estimate_motion.h:17-20:
 * cv::findEssentialMat(pts1, pts2, K, RANSAC, ransac_prob, ransac_thre, mask) + cv::recoverPose) and MotionEstimator::getDepthFast
 * (:234-283) as called per pair at cpp_code/test/sfm.cpp:163-166.  The caller gathers the matched keypoint coordinates exactly as the
 * reference does (:36-40: pts1[k] = frame_1.keypoints[matches[k].queryIdx].pt, pts2[k] = frame_2.keypoints[matches[k].trainIdx].pt), for
 * all pairs back to back: pair p owns points [pair_off[p], pair_off[p + 1]).  K is the 3 x 3 camera matrix, row-major (frame_t::K_cam):
 * one for all pairs (k_per_pair = 0) or one per pair.  Outputs: inlier_mask[k] = 1 iff match k is an inlier of the essential matrix
 * (what the reference copies into inlier_matches, :54-60), and per pair E, the recovered pose T_21 = [R | t], the inlier / cheirality
 * counts and getDepthFast's mean relative depth.  The RANSAC is OpenCV's (5-point minimal solver, Sampson error, threshold scaled by the
 * mean focal length, adaptive iteration count, first best model wins) except for its random sample sequence, which cannot be restated:
 * hypothesis h of pair p draws its five matches from a counter-based generator keyed by (seed, first_pair + p, h), so results are
 * reproducible and independent of batching.  Pairs with fewer than 5 matches, or without a model that has more than 4 inliers, get ok = 0. */
typedef struct esfm_two_view_params_t {
    double ransac_thre;       /* pixels; estimate_motion.h:20 default 1.0 (sfm.cpp passes ransac_reproj_distance) */
    double ransac_prob;       /* 0.99 */
    double cheirality_dist;   /* cv::recoverPose distanceThresh, 50 */
    uint64_t seed;
    uint64_t first_pair;      /* sampler key of pair 0 of this call (lets a caller split a job into several calls) */
    int32_t max_iters;        /* cv::findEssentialMat default 1000 */
    int32_t random_rate;      /* getDepthFast: every random_rate-th inlier, >= 1 */
} esfm_two_view_params_t;
typedef struct esfm_two_view_t {
    double E[9];              /* essential matrix, row-major, unit Frobenius norm */
    double R[9];              /* rotation of T_21, row-major */
    double t[3];              /* translation of T_21, unit length */
    double depth;             /* getDepthFast: mean norm of the triangulated inliers, in baseline lengths */
    int32_t n_matches, n_inliers, n_good;   /* n_good = inliers in front of both cameras for the chosen (R, t) */
    int32_t iters;            /* hypotheses the stopping rule evaluated */
    int32_t ok;
    int32_t reserved;
} esfm_two_view_t;
int esfm_two_view_default_params(esfm_two_view_params_t* params);
int esfm_two_view_batch(esfm_ctx_t* ctx, int64_t n_pairs, const int64_t* pair_off, const float* pts1, const float* pts2, const double* K,
                        int k_per_pair, const esfm_two_view_params_t* params, unsigned char* inlier_mask, esfm_two_view_t* out);
/* MotionEstimator::getDepthFast on its own (estimate_motion.cpp:234-283; decl estimate_motion.h:26-27, random_rate default 20): every
 * random_rate-th of the given matches (pixel coordinates, as above) triangulated with [I|0] and T_21 = [R | t]; *depth = the mean norm of the
 * points in baseline lengths, *n_used (optional) = how many were triangulated. */
int esfm_two_view_depth(esfm_ctx_t* ctx, int64_t n_matches, const float* pts1, const float* pts2, const double* K, const double* R,
                        const double* t, int random_rate, double* depth, int32_t* n_used);
/* Verification of a whole match batch, the step between matching and track building in the reference's loop (sfm.cpp:163-194).
 * `matches` is a fetched batch (ESFM_KEEP_MATCHES; a digests-only or unfetched device-resident batch -> ESFM_ERR_STATE), matched in this run
 * or loaded with esfm_results_load.  Key points: frame f owns kp_xy[2*k], kp_xy[2*k+1] for k in [kp_off[f], kp_off[f+1])
 * (frame_t::keypoints[k].pt), n_frames + 1 offsets from kp_off[0] = 0.  K: one row-major 3 x 3 for all frames (k_per_frame = 0) or one per
 * frame; a pair uses its QUERY frame's K (estimate_motion.cpp:43).  Pairs with <= min_pair_matches matches are not verified (sfm.cpp:163, 20
 * in the reference): ok = 0, no inliers, iters = 0.  Pair (i, j) draws its hypotheses from the key (i << 32) | j with params->seed -- the key
 * the C++ drop-in uses per call -- so its result does not depend on the batch, its position in it, or the device; params->first_pair must
 * be 0.  Key-point gathering, RANSAC, pose and inlier compaction run on the device; only inlier records and results return.
 * *inliers: a new batch with the same pairs in the same order, each pair's inlier records unchanged and in their original order
 * (estimate_motion.cpp:54-60), kind / ratio / cross_check / frame rows copied from `matches`; out: one record per pair.
 * ESFM_ERR_INVALID, before any output: NULL arguments, a pair outside [0, n_frames), stored frame rows (a version-2 file, or any batch the
 * library matched) that differ from the key-point counts, bad parameters (as esfm_two_view_batch), or a queryIdx / trainIdx outside its
 * frame's key points (found on the device; the message names the first such pair). */
int esfm_two_view_results(esfm_ctx_t* ctx, esfm_results_t* matches, int n_frames, const int64_t* kp_off, const float* kp_xy, const double* K,
                          int k_per_frame, const esfm_two_view_params_t* params, int min_pair_matches, esfm_results_t** inliers,
                          esfm_two_view_t* out);
/* The same on the devices of `multi`: consecutive blocks of pairs are dealt to the devices by match count, each device verifies its share with
 * its own copy of the key points, the shares are merged in the batch's pair order.  Byte-identical to esfm_two_view_results at any device
 * count (the keys are frame ids). */
int esfm_multi_two_view_results(esfm_multi_t* multi, esfm_results_t* matches, int n_frames, const int64_t* kp_off, const float* kp_xy,
                                const double* K, int k_per_frame, const esfm_two_view_params_t* params, int min_pair_matches,
                                esfm_results_t** inliers, esfm_two_view_t* out);

/* ---- ORB extraction: the step before the path (SURVEY.md section 8(f) rank 4) -------------------------------------------------------------
 * Replaces FeatureMatching::detectFeaturesORB (cpp_code/src/feature_matching.cpp:14-41; decl cpp_code/include/feature_matching.h:13, called
 * once per frame at cpp_code/test/sfm.cpp:116): cv::ORB::create(max_num)->detect(image, keypoints) followed by
 * cv::ORB::create(max_num)->compute(image, keypoints, descriptors), with OpenCV's defaults (scale factor 1.2f, 8 levels, edge threshold 31,
 * WTA_K 2, Harris score, patch size 31, FAST threshold 20).  image: 8-bit, 1 channel (gray) or 3 channels (BGR, converted as cv::cvtColor
 * does), rows x cols, row_stride bytes between rows.  The pyramid (INTER_LINEAR_EXACT), FAST-9/16 score + non-maximum suppression, Harris
 * responses, intensity-centroid angles, the 7 x 7 blur and the steered 256-bit rBRIEF tests run on the device; the host only replays
 * KeyPointsFilter::retainBest's std::nth_element / std::partition on the device-computed responses, because the order that leaves the key
 * points in is the row order of the frame's descriptors (and with it every lowest-index tie-break of the matcher).  Outputs are what cv2
 * 4.13.0 returns, bit for bit: key points in the same order with the same pt / size / angle / response / octave (class_id is always -1),
 * 32-byte descriptors.  keypoints / descriptors have room for `capacity` entries (descriptors may be NULL); ORB can return a few more than
 * max_features when Harris responses tie at the cut, so leave slack; if capacity is too small the call fails with ESFM_ERR_CAPACITY and
 * *n_out = the number needed. */
typedef struct esfm_keypoint_t {
    float x, y;               /* cv::KeyPoint::pt, full-resolution pixels */
    float size;               /* 31 * level scale */
    float angle;              /* degrees, [0, 360) */
    float response;           /* Harris response */
    int32_t octave;           /* pyramid level */
} esfm_keypoint_t;
int esfm_orb_extract(esfm_ctx_t* ctx, const unsigned char* image, int rows, int cols, int channels, size_t row_stride, int max_features,
                     esfm_keypoint_t* keypoints, unsigned char* descriptors, int capacity, int* n_out);
/* The same, with the descriptors written straight into a B256 bank that is being filled (in place of esfm_bank_set_frame): they never leave
 * the device.  descriptors_host may be NULL. */
int esfm_bank_set_frame_from_image(esfm_bank_t* bank, int frame_id, const unsigned char* image, int rows, int cols, int channels,
                                   size_t row_stride, int max_features, esfm_keypoint_t* keypoints, unsigned char* descriptors_host,
                                   int capacity, int* n_out);
/* Intermediate results of the device stages, for tests: the pyramid level `level` of the last esfm_orb_extract call on this context
 * (blurred = 0: as resized; 1: after the 7 x 7 blur), copied to out (rows * cols bytes, dense); *rows / *cols receive the level size. */
/* Host wall-clock milliseconds of the last extraction on this context: [0] upload + gray + pyramid + FAST + NMS + scan, [1] corner records
 * (Harris, angle) and their download, [2] host selection, [3] key-point upload + blur + descriptors + download, [4] the whole call;
 * *corners (optional) = NMS survivors inside the edge band, all levels. */
int esfm_orb_last_timing(esfm_ctx_t* ctx, double* phase_ms, int* corners);
int esfm_orb_debug_level(esfm_ctx_t* ctx, int level, int blurred, unsigned char* out, size_t out_bytes, int* rows, int* cols);

#ifdef __cplusplus
}
#endif
#endif /* ESFM_MATCH_H_ */
