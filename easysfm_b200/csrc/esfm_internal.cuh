// esfm_internal.cuh -- shared declarations of libesfm_match.so (sm_100a only).
//
// Data layout in HBM (see DESIGN.md "Data layout"):
//   F32X64 bank : rows_f32  float[total_rows][64]        row-major, as uploaded (used by the direct-form refinement)
//                 kmajor    float[n_tiles][64*128 + 128]  per 128-row tile: [k][row] then 128 half squared norms;
//                                                         pad rows are zeros with half-norm = +inf (self-masking)
//   B256 bank   : rows_b256 uint4[total_rows][2]          row-major 32 bytes per descriptor
//   scratch     : per pair slot 4 arrays of `stride` u64 keys: row NN1, row NN2, col NN1, col NN2
//                 key = (orderable distance bits << 32) | index ; unsigned order == (distance, lowest index)
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cfloat>

#include "../../include/esfm_match.h"

namespace esfm {

typedef unsigned long long u64;

constexpr int kDim = 64;                             // SURF descriptor length (floats)
constexpr int kTile = 128;                           // rows per k-major tile
constexpr int kTileFloats = kDim * kTile + kTile;    // 8192 operand floats + 128 half norms
constexpr int kTileBytes = kTileFloats * 4;          // 33280 B, one bulk copy
constexpr int kQTiles = 2;                           // query block = 2 tiles = 256 rows
constexpr int kConsumerThreads = 256;                // 8 consumer warps
constexpr int kSweepThreads = kConsumerThreads + 128; // + 1 producer warpgroup (only its first lane works)
constexpr u64 kKeyInit = ~0ull;
constexpr uint32_t kFltMaxBits = 0x7f7fffffu;

// ORB / Hamming sweep geometry
constexpr int kHamTile = 256;                        // train rows per smem stage (8 KB)
constexpr int kHamStages = 4;
constexpr int kHamRQ = 4;                            // query rows held in registers per thread
constexpr int kTcKindB256Z = 2;                      // internal sweep kind: B256 with the "Z" operand encoding (tc_layout.cuh)
__host__ __device__ constexpr bool tc_kind_is_f32(int k) { return k == ESFM_KIND_F32X64; }
constexpr int kTcZShift = 15;                        // Z key = kTcZ0i + (hamming << kTcZShift) + train row index inside its frame
constexpr int kTcZMaxRows = 1 << kTcZShift;          // frames with more rows use the generic tensor-core epilogue
constexpr int kTcZ0i = 21 * 448 * 448 - (1 << 22);   // 20480: what the 21 offset slots leave after cancelling -2^22
constexpr int kHamIdxBits = 20;                      // packed 32-bit key = dist << 20 | index  (rows per frame < 2^20)

// "No bound yet" of the running column thresholds: above every real value, below the pad rows.  FFMA sweep: 3.39e38f.  Tensor-core
// sweeps: SURF 7.4e28 (pads: 1e30), ORB 51015 (real 2 * hamming <= 512, pads >= 200704), ORB "Z" 1.33e7 (keys < 2^24).
constexpr uint32_t kThrInit = 0x7f7f7f7fu;
constexpr uint32_t kTcBoundBitsF32 = 0x6f6f6f6fu, kTcBoundBitsB256 = 0x47474747u, kTcBoundBitsZ = 0x4b4b4b4bu;
// Input range of the SURF engines (DESIGN.md section 5.0, "Input range"): the largest |x| of any component, M, each sweep is correct for, with
// D = kDim dims.  plan_sweep moves a bank outside an engine's range on to the next one (tc16 -> tc -> ffma); esfm_bank_commit refuses a bank
// outside ffma's.  tc16: a = fp16(x) stays finite; below kTc16MinFrameAbs in some frame, fp16's subnormal step (2^-24, the split's absolute
// error) is no longer small against that frame's distances.  tc: the largest 1/2 d^2 = 2 D M^2 = 2^95 stays below kTcBoundBitsF32 (7.4e28)
// and the pad rows (kTcPadNorm, 1e30).  ffma: D (2M)^2 = 2^126 keeps finalize's direct-form sum finite, 1/2 d^2 <= 2^125 below kThrInit.
constexpr float kTc16MaxAbs = 65504.f;
constexpr float kTc16MinFrameAbs = 0x1p-6f;
constexpr float kTcMaxAbs = 0x1p44f;
constexpr float kFfmaMaxAbs = 0x1p59f;
static_assert(2.0 * kDim * (double)kTcMaxAbs * kTcMaxAbs < 7.4e28 && 2.0 * kDim * (double)kFfmaMaxAbs * kFfmaMaxAbs < 3.39e38 &&
                  kDim * 4.0 * kFfmaMaxAbs * kFfmaMaxAbs < (double)FLT_MAX,
              "engine input ranges must stay below the column-threshold sentinels");
// cudaMemsetAsync writes the thresholds' start value, so each sentinel must be one byte repeated
__host__ __device__ constexpr bool is_byte_fill(uint32_t v) { return v == (v & 0xffu) * 0x01010101u; }
static_assert(is_byte_fill(kThrInit) && is_byte_fill(kTcBoundBitsF32) && is_byte_fill(kTcBoundBitsB256) && is_byte_fill(kTcBoundBitsZ),
              "column-threshold sentinels must be a repeated byte");

// How finalize reads the row and column keys a sweep leaves (FinalizeParams::key_format):
//   Direct  key = (distance bits << 32) | column, high word read as it is: the POPC sweep's integer Hamming distance, 1/2 d^2 of the SURF
//           ffma and tc sweeps (re-evaluated in direct form anyway);
//   TcPm1   ORB tc sweep, +-1 encoding: high word = the float 2 * hamming;
//   TcZ     ORB tc sweep, "Z" encoding: high word = the float z = kTcZ0i + 2^15 * hamming + column (tc_layout.cuh);
//   Slice   sweep_win.cu (both kinds): row keys name a slice of train columns instead of a column (see finalize.cu).
enum class KeyFormat : int { Direct, TcPm1, TcZ, Slice };

struct PairDesc {
    int32_t q_frame, t_frame;
};

struct SweepParams {
    // bank
    const float* kmajor;        // F32X64
    const uint4* rows_b256;     // B256
    const float* rows_f32;         // F32X64 row-major rows (the TC sweep converts its query tiles from these)
    const unsigned char* tc_main;  // F32X64, tensor-core engine: [tiles][69632 B] operand images (tc_layout.cuh)
    const int* frame_rows;      // [n_frames]
    const int* frame_row_off;   // [n_frames + 1]
    const int* frame_tile_off;  // [n_frames + 1]   (F32X64, in tiles)
    // work
    const PairDesc* pairs;      // device array of this chunk
    int n_pairs;
    int units_per_pair;         // query-range split factor S (>= 1)
    // scratch
    u64* keys;                  // [n_pairs][4][stride]
    uint32_t* col_thr;          // [n_pairs][stride] running column thresholds (float bits), L2 sweeps only
    int stride;                 // keys per array (>= padded rows of the largest frame in the chunk)
    int col_cap;                // Hamming sweep: smem column-minimum capacity in entries
    int tc_kind;                // TC sweeps: ESFM_KIND_F32X64 (3xTF32 L2; sweep_win: 16-bit split), ESFM_KIND_B256 (FP8 Hamming) or kTcKindB256Z (FP8 Hamming, packed
                                // (distance, column) keys from the MMA); tc_main holds that kind's images
    int need_cols;              // 0: cross_check is off, nobody reads the column minima -- the tensor-core sweeps skip the column side
    // sweep_win.cu, verification pass of the two-phase cross-check: the query operand is a GATHERED subset of the pair's TRAIN frame
    // (gather[pair * stride + slot] = row of the train frame, gather_cnt[pair] rows), swept against the pair's QUERY frame; the best
    // (value, slice) of every gathered row lands in the pair's 4th key array at [slot].  NULL = a normal sweep.
    const int* gather;
    const int* gather_cnt;
    // SURF (sweep_win.cu): 1 = FAST mode, the query enters as a = fp16(x) only: 8 kind::f16 MMAs + the norm step = 9 slots per tile instead
    // of 13, values within win_fast_eps of the exact ones.  0 = exact mode (13 slots).
    int win_fast;
    // with `gather`: 1 = FALLBACK sweep, the gathered rows are rows of the pair's QUERY frame (the ones the fast sweep could not settle),
    // swept in exact mode against the pair's train frame; their (best, second) keys overwrite rk1 / rk2 at the original row, marked with
    // kWinExactMark.  0 = the role-swapped verification sweep above.
    int fallback;
    int debug_flags;            // TC sweep pipeline probes ($ESFM_TC_DEBUG; results are WRONG when set): 1 = epilogue only drains,
                                // 2 = no MMAs issued, 4 = no train-tile loads, 8 = no column events, 16 = no row selection, 32 = column events without their atomics, 64 = column events found but not handled
};

struct FinalizeParams {
    int kind;
    const float* rows_f32;
    const uint4* rows_b256;
    const int* frame_rows;
    const int* frame_row_off;
    const PairDesc* pairs;
    int n_pairs;
    u64* keys;
    int stride;
    double ratio;
    int cross_check;
    esfm_dmatch_t* arena;       // dense match arena
    unsigned long long arena_cap;
    unsigned long long* cursor; // arena allocation cursor (matches)
    unsigned long long* pair_off;  // [n_pairs] offset of each pair's matches in the arena
    int32_t* pair_cnt;          // [n_pairs]
    int* overflow;              // set to 1 if the arena was too small
    KeyFormat key_format;
    int phase;                  // 0 = everything in one launch; two-phase cross-check (finalize.cu): 1 = ratio test + list of the train rows to verify,
                                // 2 = verdicts of the verification sweep + compaction
    int* gather;                // [n_pairs][stride] phase 1 out / the verification sweep's input
    int* gather_cnt;            // [n_pairs]
    // SURF rows from the FAST sweep (SweepParams::win_fast; NULL = every row was swept in exact mode): per bank row |x - fp16(x)|_2,
    // per frame the largest |x|_2 (launch_pack_tch) -> win_fast_eps.  Rows whose key carries kWinExactMark were re-swept exactly.
    // frame_norm is also set in exact mode: phase 1 of the two-phase cross-check scales its margin with it.
    const float* row_eps;
    const float* frame_norm;
    unsigned long long* fallback_rows;   // win_classify: += rows put on the fallback list
    unsigned long long* verified_rows;   // two-phase cross-check, phase 1: += train rows put on the verification list
    // optional raw knn output for one pair (esfm_knn2_pair)
    int32_t* knn_idx;
    float* knn_dist;
};

// ---- host-side launchers (defined in the .cu files) -------------------------------------------
cudaError_t launch_pack_f32(const float* rows, const int* frame_rows, const int* frame_row_off, const int* frame_tile_off,
                            int n_frames, int n_tiles_total, float* kmajor, cudaStream_t s);
cudaError_t launch_pack_tc8(const uint32_t* rows, const int* frame_rows, const int* frame_row_off, const int* frame_tile_off,
                            int n_frames, int n_tiles_total, unsigned char* tc_main, int z_mode, cudaStream_t s);
cudaError_t launch_pack_tc(const float* rows, const int* frame_rows, const int* frame_row_off, const int* frame_tile_off,
                           int n_frames, int n_tiles_total, unsigned char* tc_main, cudaStream_t s);
cudaError_t launch_pack_tch(const float* rows, const int* frame_rows, const int* frame_row_off, const int* frame_tile_off,
                            int n_frames, int n_tiles_total, unsigned char* tc_main, float* row_eps, float* frame_norm, cudaStream_t s);
cudaError_t launch_frame_absmax(const float* rows, const int* frame_rows, const int* frame_row_off, const int* frame_tile_off, int n_frames,
                                int n_tiles_total, unsigned* frame_absmax, cudaStream_t s);
cudaError_t launch_sweep_l2(const SweepParams& p, int sm_count, cudaStream_t s);
cudaError_t launch_sweep_win(const SweepParams& p, int sm_count, cudaStream_t s);
cudaError_t launch_sweep_l2_tc(const SweepParams& p, int sm_count, cudaStream_t s);
cudaError_t launch_sweep_hamming(const SweepParams& p, int sm_count, cudaStream_t s);
cudaError_t launch_finalize(const FinalizeParams& p, cudaStream_t s);
cudaError_t launch_win_classify(const FinalizeParams& p, cudaStream_t s);
size_t sweep_l2_smem_bytes(int stages);
size_t sweep_hamming_smem_bytes(int col_cap);
int sweep_l2_max_rows();       // largest frame (rows) the L2 sweep supports
int sweep_hamming_max_rows();

// Low-word bit of a slice key (sweep_win.cu) whose row was swept in exact mode by the fallback sweep (slice ids stay below 2^30).
constexpr uint32_t kWinExactMark = 0x80000000u;

// ---- device helpers ------------------------------------------------------------------------------
#ifdef __CUDACC__
// Bound on |v' - v| for every train row t of a frame, v' = what the FAST SURF sweep ranks by (a_q.(a_t + b_t) - 1/2|q|^2 - 1/2|t|^2 in
// fp32 accumulation, a = fp16(x), b = fp16(x - a)), v = -1/2 |q - t|^2 exactly (DESIGN.md section 5.0, "the fast-mode bound"):
//     v' - v = -(q - a_q).t - a_q.r_t + rounding,    r_t = t - a_t - b_t,   |r_t| <= 2^-22 |t| + 2^-22 (64 dims, fp16 subnormals)
// e_q = |q - a_q|_2, n_q / n_t = the largest row norms of the query / train frame (all rounded up).  The last term covers the fp32 sums
// of the two half norms (2 x 64 fused steps) and the 9 MMA accumulations (17 addends each, truncated, none above m).
// (Written with the _rn intrinsics, which the compiler never contracts: win_classify_kernel and finalize must compute the same bits.)
__device__ __forceinline__ float win_fast_eps(float e_q, float n_q, float n_t) {
    const float m = __fadd_rn(__fmul_rn(0.5f, __fadd_rn(__fmul_rn(n_q, n_q), __fmul_rn(n_t, n_t))), __fmul_rn(n_q, n_t));
    const float r = __fmul_rn(__fadd_rn(n_q, e_q), __fmul_rn(0x1p-22f, __fadd_rn(n_t, 1.f)));
    return __fmul_rn(__fadd_rn(__fadd_rn(__fmul_rn(e_q, n_t), r), __fmul_rn(0x1p-15f, m)), 1.001f);
}
// Ratio test on the sweep's 1/2 d^2 values s1 <= s2 of a row whose every value is within e of the exact one (e = 0: an exact-mode
// sweep, whose own ~4e-7 is what the 0.1 % + 4e-6 margins absorb): 0 = fails for certain, 1 = passes for certain (and for e > 0 no other
// column can be the nearest: the best slice holds it), 2 = to be decided on exact distances.  SURF chain keys (sweep_win.cu): s2 is the best
// value OUTSIDE the best chain, an upper bound on the true second (+inf: no second chain), so 0 stays certain and 1 speaks for the columns
// outside the best chain only: finalize tests the best chain's own second exactly.
__device__ __forceinline__ int win_ratio_class(float s1, float s2, float e, float r2) {
    if (__fsub_rn(s1, e) > __fadd_rn(__fmul_rn(__fmul_rn(r2, __fadd_rn(s2, e)), 1.001f), 4e-6f)) return 0;
    if (__fadd_rn(s1, e) < __fsub_rn(__fmul_rn(__fmul_rn(r2, __fsub_rn(s2, e)), 0.999f), 4e-6f) && (e == 0.f || __fsub_rn(s2, s1) > 2.f * e)) return 1;
    return 2;
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// Arrive WITHOUT release semantics.  A releasing arrive first waits until the thread's earlier memory operations have been
// performed -- including fire-and-forget global atomics (RED) on their way to L2, a round trip of a thousand cycles under load.
// The tensor-core epilogue posts column minima with such atomics and then frees pipeline stages whose contents it has ALREADY
// consumed (tcgen05.wait::ld has returned / the loaded thresholds have been compared): nothing the consumer of the barrier reads
// depends on those atomics, so the arrive needs no ordering with them.
__device__ __forceinline__ void mbar_arrive_relaxed(uint64_t* bar) {
    asm volatile("mbarrier.arrive.relaxed.cta.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    while (!mbar_try_wait(bar, parity)) {
    }
}
// Producer-side wait: the ring has slack, so sleep between polls instead of burning issue slots of the
// SM sub-partition the producer warp shares with two consumer warps.
__device__ __forceinline__ void mbar_wait_backoff(uint64_t* bar, uint32_t parity) {
    uint32_t ok = 0;
    while (true) {
        // try_wait with a suspend-time hint: the hardware may park the thread until the phase completes
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok)
            : "r"(smem_u32(bar)), "r"(parity), "r"(1000000u)
            : "memory");
        if (ok) break;
        __nanosleep(2000);
    }
}
// TMA 1-D bulk copy global -> shared, completion signalled on an mbarrier (SASS: UBLKCP).
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(smem_dst)),
                 "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
// Register rebalancing between warpgroups (setmaxnreg works on 4-warp groups): the 384-thread CTA is
// launched at 168 regs/thread; the producer group drops to 40 and the two consumer groups grow to 232.
template <int N> __device__ __forceinline__ void reg_dealloc() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N)); }
template <int N> __device__ __forceinline__ void reg_alloc() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N)); }
// named barrier over the consumer warps only (the producer warp never joins)
__device__ __forceinline__ void consumer_sync() { asm volatile("bar.sync 1, %0;" ::"n"(kConsumerThreads) : "memory"); }

__device__ __forceinline__ u64 make_key(uint32_t hi, uint32_t idx) { return ((u64)hi << 32) | idx; }

// 256-bit read-only global load (sm_100: LDG.E.256): half as many load instructions -- and L1 tag lookups -- per
// gathered descriptor row as float4 loads.  `p` must be 32-byte aligned (descriptor rows are 256 bytes).
struct __align__(32) float8 { float v[8]; };
__device__ __forceinline__ float8 ldg256(const float* p) {
    float8 r;
    asm("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=f"(r.v[0]), "=f"(r.v[1]), "=f"(r.v[2]), "=f"(r.v[3]), "=f"(r.v[4]), "=f"(r.v[5]), "=f"(r.v[6]), "=f"(r.v[7])
                 : "l"(p));
    return r;
}

// Direct-form squared-difference distance with the summation order fixed in oracle/bf_oracle.c:
// four partial sums over dims j = l (mod 4), fused multiply-add, (s0+s1)+(s2+s3), IEEE sqrt.
__device__ __forceinline__ float l2_direct(const float* __restrict__ a, const float* __restrict__ b) {
    float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
#pragma unroll
    for (int c = 0; c < kDim / 8; ++c) {
        const float8 x = ldg256(a + 8 * c), y = ldg256(b + 8 * c);
#pragma unroll
        for (int h = 0; h < 2; ++h) {      // dims 8c + 4h .. 8c + 4h + 3, in ascending order as the oracle sums them
            const float t0 = __fsub_rn(x.v[4 * h], y.v[4 * h]), t1 = __fsub_rn(x.v[4 * h + 1], y.v[4 * h + 1]);
            const float t2 = __fsub_rn(x.v[4 * h + 2], y.v[4 * h + 2]), t3 = __fsub_rn(x.v[4 * h + 3], y.v[4 * h + 3]);
            s0 = __fmaf_rn(t0, t0, s0);
            s1 = __fmaf_rn(t1, t1, s1);
            s2 = __fmaf_rn(t2, t2, s2);
            s3 = __fmaf_rn(t3, t3, s3);
        }
    }
    return __fsqrt_rn(__fadd_rn(__fadd_rn(s0, s1), __fadd_rn(s2, s3)));
}
#endif  // __CUDACC__

}  // namespace esfm
