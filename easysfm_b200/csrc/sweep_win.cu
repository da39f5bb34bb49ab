// sweep_win.cu -- round-2 tensor-core sweeps with WINDOW keys (sm_100a): half the tensor-pipe time and half the operand bytes of
// sweep_l2_tc.cu, and a selection epilogue that carries no column indices.
//
// Same contract towards the caller as the other sweeps (cpp_code/src/feature_matching.cpp:71-92 / :115-137 as exact brute force,
// python_code/feature_match.py:26-27,33-39): per image pair the two nearest train rows of every query row and the nearest query
// row of every train row, with OpenCV's lowest-index tie-break.  What differs is HOW a row's neighbours are reported:
//     row key    = value bits << 32 | SLICE,    slice = (first column / 8) << 2 | width code: the 8, 32 or 64 train columns the value
//                                               was found in (SURF: CHAIN keys, the best chain of 8 columns and the second chain of 8)
//     column key = value bits << 32 | query row                                                    (unchanged)
// finalize.cu finds the column inside the window by re-evaluating its distances exactly (direct-form L2 / XOR + POPC), which it
// only does for the rows that can pass the ratio test.  The epilogue therefore needs VALUES only:
//   * SURF (KIND = ESFM_KIND_F32X64, "H" split of tc_layout.cuh): 12 x tcgen05.mma.kind::f16 (a = fp16(x), b = fp16(x - a);
//     b_q.a_t + a_q.b_t + a_q.a_t, fp32 accumulation; fp16 subnormals are honoured by the tensor core: h16_probe.cu) + the exact
//     kind::tf32 half-norm step = 13 MMA slots per 128 x 128 tile instead of 25, tile image 36 KB instead of 68 KB.  FAST mode
//     (SweepParams::win_fast, the rows-only sweep's default) drops b_q: 8 + 1 = 9 slots, values within win_fast_eps (esfm_internal.cuh);
//     the rows that bound cannot settle are swept again in exact mode (SweepParams::fallback, finalize.cu win_classify_kernel).  Epilogue:
//     chain keys -- the maximum of every chain of 8 columns (FMNMX3), the two largest of a unit's 8 chain maxima with their chains, merged
//     into the running (k1, w1, k2, w2): ~1.2 ALU instructions per comparison instead of ~3 for an exact per-row top 2.  The row's true
//     second lies in its best chain or is its second chain's maximum; finalize evaluates the best chain exactly and learns the rest.
//   * ORB (KIND = ESFM_KIND_B256): the +-1 FP8 operands of sweep_l2_tc.cu with FP16 ACCUMULATORS (-2 hamming, exact; pad rows
//     overflow to -inf): tcgen05.ld.pack::16b delivers two columns per register and the whole epilogue runs on packed halves
//     (HMNMX2 / VHMNMX tournament, HFMA2.RELU threshold tests): ~1/2 the instructions per element of the fp32 epilogue.
// The kernel is ROWS-ONLY: the cross-check is decided by finalize.cu from the row results (claims + histograms), and the train rows that
// remain undecided are swept once more through this same kernel with the roles swapped and the query operand gathered
// (SweepParams::gather).  Raw knn output (esfm_knn2_pair) needs column minima: it runs on sweep_l2_tc.cu.
//
// Pipeline: one persistent CTA per SM, 24 warps --
//   warp 16      TMA producer: one cp.async.bulk per 36 KB train tile image into a 5-stage ring;
//   warps 17-19  MMA issuers, tile g belongs to issuer g % 3 (the tcgen05.mma queue is shallow: while one issuer is blocked in its
//                burst of MMAs the next has already passed its barrier waits -- one issuer left the tensor pipe dry ~45 % of the time,
//                csrc/microbench/pipe_probe.cu); query operand in tensor memory, 3 accumulator stages of 128 columns;
//   warps 20-23  query writers (rows of the query tile -> operand columns of tensor memory, augmented block in shared memory);
//   warps 0-15   epilogue in four GROUPS of four warps (one per TMEM lane quarter = 32 query rows).  The unit of work is half a tile
//                (64 train columns): unit 2 g + h belongs to group (2 g + h) % 4, so a group reads one half of every other tile -- ORB: 32
//                packed registers in one tcgen05.ld; SURF: two loads of 32 -- releases its share of the accumulator stage BEFORE it
//                computes, and runs one selection over its columns: twice the columns per barrier hand-shake and per running-state
//                merge of a 32-column pass, and a slow warp delays nobody else's stage.
// Every mbarrier keeps ONE producer and ONE consumer role (a parity wait may not skip a phase): the barriers of the load ring are indexed
// by tile % lcm(5 stages, 3 issuers) = 15, those of the accumulator ring by tile % lcm(3 stages, 3 issuers, 4 groups) = 12.
#include <cuda_fp16.h>

#include "tc_sweep_common.cuh"

namespace esfm {

namespace {

constexpr int kWinStages = 5;                       // shared-memory train stages (36 KB each)
// MMA issuers: the tcgen05.mma queue is shallow, so the tensor pipe runs dry while ONE issuer thread does a tile's book-keeping (two barrier
// waits, two commits: ~500 clk against 577 / 833 clk of MMAs per tile; csrc/microbench/pipe_probe.cu).  Three warps take the tiles in turn:
// while one is blocked issuing its MMAs the next has already passed its waits.  Every barrier must keep ONE issuer (a parity wait may not
// skip a phase): the accumulator ring has 3 stages = 3 issuers; the load ring indexes its barriers by tile % lcm(stages, issuers).
constexpr int kWinIssuers = 3;
constexpr int kWinLoadBars = 15;                    // lcm(kWinStages, kWinIssuers)
static_assert(kWinLoadBars % kWinStages == 0 && kWinLoadBars % kWinIssuers == 0, "load-ring barriers");
constexpr int kWinAccStages = 3;                    // (512 - 64) / 128 accumulator stages
constexpr uint32_t kWinACol0 = 128u * kWinAccStages; // query operand: 64 tensor-memory columns (SURF: a 32 | b 32; ORB: 256 FP8)
constexpr int kWinTileBytes = kTchTileBytes;        // == kTc8TileBytes
constexpr int kWinMainBytes = kTchMainBytes;
constexpr int kWinGroupBytes = kTchGroupBytes;
static_assert(kTchTileBytes == kTc8TileBytes && kTchMainBytes == kTc8MainBytes && kTchGroupBytes == kTc8GroupBytes, "the two kinds share one geometry");
constexpr int kWinGroups = 4;                       // epilogue groups (4 warps each); tile g belongs to group g % 4
constexpr int kWinAccBars = 12;                     // lcm(kWinAccStages, kWinIssuers, kWinGroups)
static_assert(kWinAccBars % kWinAccStages == 0 && kWinAccBars % kWinIssuers == 0 && kWinAccBars % kWinGroups == 0, "accumulator-ring barriers");
constexpr float kWinNone = -3.0e38f;                // "no candidate": below every real value and every pad
// slice ids of the row keys: (first column / 8) << 2 | width code (0: 8 columns, 1: 32, 2: 64, 3: 128) -- finalize.cu win_range
__device__ __forceinline__ int win_slice(int first_col, int wcode) { return ((first_col >> 3) << 2) | wcode; }

__device__ __forceinline__ uint32_t hmax2(uint32_t a, uint32_t b) { uint32_t r; asm("max.f16x2 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b)); return r; }
__device__ __forceinline__ uint32_t hmin2(uint32_t a, uint32_t b) { uint32_t r; asm("min.f16x2 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b)); return r; }
__device__ __forceinline__ float h_lo(uint32_t x) { return __low2float(*reinterpret_cast<const __half2*>(&x)); }
__device__ __forceinline__ float h_hi(uint32_t x) { return __high2float(*reinterpret_cast<const __half2*>(&x)); }
// 32 lanes x 64 consecutive columns of fp16 accumulators, two columns per register
__device__ __forceinline__ void tmem_ld32_pack(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.pack::16b.b32 "
        "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
          "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]),
          "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]),
          "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr)
        : "memory");
}

// merge a unit's two largest values (p1 >= p2, found in the column slices id1 / id2) into the running (k1, w1, k2, w2): strict
// comparisons, so of equal values the one found first (the lower slice = the lower column) stays in front
__device__ __forceinline__ void win_merge(float p1, int id1, float p2, int id2, float& k1, int& w1, float& k2, int& w2) {
    const bool c1 = p1 > k1;
    const float nk2 = fmaxf(c1 ? p2 : k2, fminf(k1, p1));
    const int wa = p2 > k1 ? id2 : w1;           // (c1)  second = p2 (this pass) or the demoted old best
    const int wb = p1 > k2 ? id1 : w2;           // (!c1) second = p1 (this pass) or unchanged
    w2 = c1 ? wa : wb;
    k2 = nk2;
    w1 = c1 ? id1 : w1;
    k1 = fmaxf(k1, p1);
}

// work decoding: a normal sweep takes (query frame, train frame) from the pair list; the verification sweep of the two-phase
// cross-check swaps the roles and reads its query rows through the pair's gather list; the fallback sweep reads them through the list
// without swapping
struct WinUnit {
    int pair, q_frame, t_frame;
    int fq;              // query rows of this unit's pair (gathered rows in a verification sweep)
    int ntt;
    int qb0, qb1;        // query TILES [qb0, qb1) of this unit
};
__device__ __forceinline__ WinUnit win_decode_unit(const SweepParams& p, int unit) {
    WinUnit u;
    u.pair = unit / p.units_per_pair;
    const int part = unit - u.pair * p.units_per_pair;
    const PairDesc pd = p.pairs[u.pair];
    int nqt;
    if (p.gather) {
        u.q_frame = p.fallback ? pd.q_frame : pd.t_frame;
        u.t_frame = p.fallback ? pd.t_frame : pd.q_frame;
        u.fq = p.gather_cnt[u.pair];
        nqt = (u.fq + kTile - 1) / kTile;
    } else {
        u.q_frame = pd.q_frame;
        u.t_frame = pd.t_frame;
        u.fq = p.frame_rows[pd.q_frame];
        nqt = p.frame_tile_off[pd.q_frame + 1] - p.frame_tile_off[pd.q_frame];
    }
    u.ntt = p.frame_tile_off[u.t_frame + 1] - p.frame_tile_off[u.t_frame];
    u.qb0 = (int)((long long)nqt * part / p.units_per_pair);
    u.qb1 = (int)((long long)nqt * (part + 1) / p.units_per_pair);
    if (p.frame_rows[u.t_frame] < 1) u.qb1 = u.qb0;
    return u;
}

}  // namespace

template <int KIND>
__global__ void __launch_bounds__(kTcThreads, 1) sweep_win_kernel(const SweepParams p) {
    constexpr bool kOrb = KIND != ESFM_KIND_F32X64;
    extern __shared__ unsigned char smem_raw[];
    unsigned char* base = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);       // SWIZZLE_128B atoms: 1024-byte alignment
    unsigned char* Ts = base;                                   // kWinStages train tile images (36 x 1024 B each)
    unsigned char* Qa = Ts + kWinStages * kWinTileBytes;        // augmented block of the query tile
    u64* mkey = reinterpret_cast<u64*>(Qa + kTcAugBytes);       // [best, second][128] merged row keys
    uint64_t* bars = reinterpret_cast<uint64_t*>(mkey + 2 * kTile);
    uint64_t* fullQ = bars;
    uint64_t* fullT = fullQ + 1;
    uint64_t* emptyT = fullT + kWinLoadBars;
    uint64_t* accFull = emptyT + kWinLoadBars;
    uint64_t* accEmpty = accFull + kWinAccBars;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(accEmpty + kWinAccBars);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n_units = p.n_pairs * p.units_per_pair;
    const bool nosleep = (p.debug_flags & 128) != 0;      // probe: the producer / issuers poll their barriers without sleeping

    if (threadIdx.x == 0) {
        mbar_init(&fullQ[0], 4);                      // the 4 query-writer warps
        for (int s = 0; s < kWinLoadBars; ++s) {
            mbar_init(&fullT[s], 1);
            mbar_init(&emptyT[s], 1);                 // MMA commit
        }
        for (int s = 0; s < kWinAccBars; ++s) {
            mbar_init(&accFull[s], 1);                // MMA commit
            mbar_init(&accEmpty[s], 8);               // the 4 + 4 warps of the two epilogue groups that own the tile's halves
        }
        fence_mbar_init();
    }
    if (warp == kTcEpiWarps + 1) tmem_alloc(tmem_slot, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;

    if (warp >= kTcEpiWarps) {
    reg_dealloc<kTcServiceRegs>();
    if (warp == kTcEpiWarps) {
        // ======================= TMA producer =======================
        if (lane == 0) {
            uint32_t g = 0;
            for (int unit = blockIdx.x; unit < n_units; unit += gridDim.x) {
                const WinUnit u = win_decode_unit(p, unit);
                const unsigned char* timg = p.tc_main + (size_t)p.frame_tile_off[u.t_frame] * kWinTileBytes;
                for (int qt = u.qb0; qt < u.qb1; ++qt) {
                    for (int tt = 0; tt < u.ntt; ++tt, ++g) {
                        // stage g % 5, its barrier pair g % 15; the stage was last read by tile g - 5 (barrier (g - 5) % 15)
                        const uint32_t st = g % kWinStages, bi = g % kWinLoadBars;
                        if (g >= kWinStages) {
                            const uint32_t pg = g - kWinStages, pbi = pg % kWinLoadBars, pph = (pg / kWinLoadBars) & 1;
                            if (nosleep) mbar_wait_sleep<0>(&emptyT[pbi], pph); else mbar_wait_sleep<kTcSleepProducer>(&emptyT[pbi], pph);
                        }
                        mbar_arrive_expect_tx(&fullT[bi], kWinTileBytes);
                        if (p.debug_flags & 4)
                            asm volatile("mbarrier.complete_tx.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(&fullT[bi])), "r"(kWinTileBytes) : "memory");
                        else
                            bulk_g2s(Ts + (size_t)st * kWinTileBytes, timg + (size_t)tt * kWinTileBytes, kWinTileBytes, &fullT[bi]);
                    }
                }
            }
        }
    } else if (warp >= kTcEpiWarps + 1 && warp <= kTcEpiWarps + kWinIssuers) {
        // ======================= MMA issuers (warp-uniform control flow, one elected lane issues): tile g belongs to issuer g % 3 =======================
        const uint32_t me = (uint32_t)(warp - (kTcEpiWarps + 1));
        constexpr uint32_t id_main = kOrb ? tc_idesc_e4m3_h(128, 128) : tc_idesc_f16(128, 128, 0, 0);
        const uint64_t qad = tc_desc_nosw(smem_u32(Qa), 128, kTcAugGroupBytes);
        const uint64_t td0 = tc_desc_sw128(smem_u32(Ts), kWinGroupBytes);
        const uint64_t tad0 = tc_desc_nosw(smem_u32(Ts) + kWinMainBytes, 128, kTcAugGroupBytes);
        uint32_t g = 0, qn = 0;
        for (int unit = blockIdx.x; unit < n_units; unit += gridDim.x) {
            const WinUnit u = win_decode_unit(p, unit);
            for (int qt = u.qb0; qt < u.qb1; ++qt, ++qn) {
                // every issuer observes every fill of the query slot (a parity wait may not skip a phase), also in a block none of whose
                // tiles are its own
                mbar_wait_sleep<0>(&fullQ[0], qn & 1);
                for (int tt = 0; tt < u.ntt; ++tt, ++g) {
                    if (g % kWinIssuers != me) continue;
                    const uint32_t st = g % kWinStages, bi = g % kWinLoadBars, ph = (g / kWinLoadBars) & 1;
                    if (nosleep) mbar_wait_sleep<0>(&fullT[bi], ph); else mbar_wait_sleep<kTcSleepIssuer>(&fullT[bi], ph);
                    const uint64_t td = td0 + (uint64_t)(st * (kWinTileBytes >> 4));
                    const uint64_t tad = tad0 + (uint64_t)(st * (kWinTileBytes >> 4));
                    const uint32_t as = g % kWinAccStages, ab = g % kWinAccBars;
                    if (g >= kWinAccStages) {          // the accumulator stage was last used by tile g - 3: its group must have read it
                        const uint32_t pg = g - kWinAccStages, pab = pg % kWinAccBars, pph = (pg / kWinAccBars) & 1;
                        if (nosleep) mbar_wait_sleep<0>(&accEmpty[pab], pph); else mbar_wait_sleep<kTcSleepIssuer>(&accEmpty[pab], pph);
                    }
                    tc_fence_after();
                    const uint32_t d = tmem + as * 128;
                    const uint32_t acol = tmem + kWinACol0;
                    if (!(p.debug_flags & 2) && elect_one()) {
                        if (kOrb) {
                            // 256 FP8 values per row = 8 k-steps of K = 32 (32 bytes each): v = 256 - 2 hamming.  (No augmented step: the
                            // pad columns of a frame's last tile are masked in the epilogue.)
#pragma unroll
                            for (int ks = 0; ks < 8; ++ks)
                                tc_mma_f8_ts(d, acol + ks * 8, td + (uint64_t)(((ks >> 2) * 1024 + (ks & 3) * 32) >> 4), id_main, ks > 0);
                        } else {
                            // small terms first: b_q.a_t (exact mode only), a_q.b_t, then a_q.a_t; a k-step = 16 halves = 32 bytes of the
                            // 128-byte row
                            if (!p.win_fast) {
#pragma unroll
                                for (int ks = 0; ks < 4; ++ks) tc_mma_f16_ts(d, acol + 32 + ks * 8, td + (uint64_t)((ks * 32) >> 4), id_main, ks > 0);
                            }
#pragma unroll
                            for (int ks = 0; ks < 4; ++ks)
                                tc_mma_f16_ts(d, acol + ks * 8, td + (uint64_t)((1024 + ks * 32) >> 4), id_main, ks > 0 || !p.win_fast);
#pragma unroll
                            for (int ks = 0; ks < 4; ++ks) tc_mma_f16_ts(d, acol + ks * 8, td + (uint64_t)((ks * 32) >> 4), id_main, true);
                            tc_mma_tf32(d, qad, tad, tc_idesc_tf32(128, 128), true);   // - 1/2|q|^2 - 1/2|t|^2, exact
                        }
                    }
                    __syncwarp();
                    if (elect_one()) {
                        tc_commit(&accFull[ab]);        // accumulator stage ready for its epilogue group
                        tc_commit(&emptyT[bi]);         // shared-memory stage consumed
                    }
                    __syncwarp();
                }
            }
        }
    } else if (warp >= kTcWriterWarp0) {
        // ======================= query writers: rows of the query tile -> operand columns of tensor memory =======================
        const int quarter = warp & 3;
        const int trow = quarter * 32 + lane;
        const uint32_t lane_addr = (uint32_t)(quarter * 32) << 16;
        const uint32_t acol = tmem + lane_addr + kWinACol0;
        unsigned char* qa = Qa + (trow >> 3) * kTcAugGroupBytes + (trow & 7) * 16;
        uint32_t quse = 0;
        int prev_last = 0;          // how many epilogue warps arrive for the block filled last: min(3, its train tiles), see the epilogue
        for (int unit = blockIdx.x; unit < n_units; unit += gridDim.x) {
            const WinUnit u = win_decode_unit(p, unit);
            const int fq = u.fq;
            const int* gl = p.gather ? p.gather + (size_t)u.pair * p.stride : nullptr;
            for (int qt = u.qb0; qt < u.qb1; ++qt) {
                const int slot = qt * kTile + trow;
                const bool valid = slot < fq;
                const int r = (gl && valid) ? __ldg(gl + slot) : slot;      // verification sweep: the slot's row of the (original) train frame
                if (kOrb) {
                    const uint4* qbits = p.rows_b256 + (size_t)p.frame_row_off[u.q_frame] * 2;
                    uint4 w0 = make_uint4(0u, 0u, 0u, 0u), w1 = w0;
                    if (valid) { w0 = __ldg(qbits + (size_t)r * 2); w1 = __ldg(qbits + (size_t)r * 2 + 1); }
                    // The slot is free once every MMA that read the previous tile has retired: the writers block on NAMED BARRIER 2,
                    // which the epilogue groups arrive at when they have seen the block's last accumulators complete.
                    if (quse > 0) named_bar_sync(2, 128 + 32 * prev_last);
                    ++quse;
                    tc_fence_after();
                    *reinterpret_cast<uint4*>(qa) = make_uint4((valid ? 0u : kFp8Pos448) | (kFp8Pos448 << 8) | (kFp8Pos16 << 16), 0u, 0u, 0u);
                    *reinterpret_cast<uint4*>(qa + 128) = make_uint4(0u, 0u, 0u, 0u);
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                    const uint32_t ws[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
#pragma unroll
                    for (int m = 0; m < 8; ++m) {       // word m = elements 32 m .. 32 m + 31 = 8 columns
                        uint32_t c[8];
#pragma unroll
                        for (int j = 0; j < 8; ++j) c[j] = valid ? tc8_expand4(ws[m] >> (4 * j)) : 0u;
                        tmem_st8(acol + m * 8, c);
                    }
                } else {
                    const float4* xr = reinterpret_cast<const float4*>(p.rows_f32 + (size_t)p.frame_row_off[u.q_frame] * kDim) + (size_t)(valid ? r : 0) * 16;
                    // pass 1: 1/2|q|^2 in the summation order of bank.cu's pack kernels
                    float hs = 0.f;
#pragma unroll 4
                    for (int m = 0; m < 16; ++m) {
                        const float4 x = __ldg(xr + m);
                        hs = __fmaf_rn(x.x, x.x, hs); hs = __fmaf_rn(x.y, x.y, hs);
                        hs = __fmaf_rn(x.z, x.z, hs); hs = __fmaf_rn(x.w, x.w, hs);
                    }
                    const float hq = valid ? 0.5f * hs : kTcPadNorm;       // pad rows can never win a column
                    float hqh, hqm, hql;
                    tc_split3(hq, hqh, hqm, hql);
                    if (quse > 0) named_bar_sync(2, 128 + 32 * prev_last);
                    ++quse;
                    tc_fence_after();
                    *reinterpret_cast<float4*>(qa) = make_float4(1.f, 1.f, 1.f, hqh);
                    *reinterpret_cast<float4*>(qa + 128) = make_float4(hqm, hql, 0.f, 0.f);
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                    // pass 2: the row again (L1/L2 hit), 16 dims at a time -> 8 columns of a (fp16 pairs) and, in exact mode, 8 of b
#pragma unroll 1
                    for (int m = 0; m < 4; ++m) {
                        uint32_t ca[8], cb[8];
#pragma unroll
                        for (int h = 0; h < 4; ++h) {
                            float4 x = __ldg(xr + 4 * m + h);
                            if (!valid) x = make_float4(0.f, 0.f, 0.f, 0.f);
                            const __half2 a0 = __floats2half2_rn(x.x, x.y), a1 = __floats2half2_rn(x.z, x.w);
                            ca[2 * h] = *reinterpret_cast<const uint32_t*>(&a0); ca[2 * h + 1] = *reinterpret_cast<const uint32_t*>(&a1);
                            if (!p.win_fast) {
                                const float2 f0 = __half22float2(a0), f1 = __half22float2(a1);
                                const __half2 b0 = __floats2half2_rn(x.x - f0.x, x.y - f0.y), b1 = __floats2half2_rn(x.z - f1.x, x.w - f1.y);
                                cb[2 * h] = *reinterpret_cast<const uint32_t*>(&b0); cb[2 * h + 1] = *reinterpret_cast<const uint32_t*>(&b1);
                            }
                        }
                        tmem_st8(acol + m * 8, ca);
                        if (!p.win_fast) tmem_st8(acol + 32 + m * 8, cb);
                    }
                }
                tmem_st_wait();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&fullQ[0]);
                prev_last = u.ntt < kWinIssuers ? u.ntt : kWinIssuers;
            }
        }
        if (quse > 0) named_bar_sync(2, 128 + 32 * prev_last);      // the epilogue arrives once per block; the last arrival has no refill waiting
    }
    } else {
        // ======================= epilogue warps: group = warp / 4 owns the tiles g % 4 == group =======================
        reg_alloc<kTcEpiRegs>();
        const int quarter = warp & 3, group = warp >> 2;
        const int trow = quarter * 32 + lane;               // row inside the 128-row query tile (= TMEM lane)
        const uint32_t lane_addr = (uint32_t)(quarter * 32) << 16;
        if (group == 0) {
            mkey[trow] = kKeyInit;
            mkey[kTile + trow] = kKeyInit;
        }
        asm volatile("bar.sync 1, %0;" ::"n"(kTcEpiThreads) : "memory");
        uint32_t g = 0;
        for (int unit = blockIdx.x; unit < n_units; unit += gridDim.x) {
            const WinUnit u = win_decode_unit(p, unit);
            u64* rk1 = p.keys + (size_t)u.pair * 4 * p.stride;
            u64* rk2 = rk1 + p.stride;
            const int ft = p.frame_rows[u.t_frame];
            // The query slot may be refilled once every MMA of the block has completed.  MMAs of ONE issuer complete in issue order, so
            // the block's last min(3, tiles) tiles -- the last tile of every issuer -- cover all of them: the quarter-0 warp of each
            // such tile's group arrives at the writers' named barrier.
            const int n_last = u.ntt < kWinIssuers ? u.ntt : kWinIssuers;
            for (int qt = u.qb0; qt < u.qb1; ++qt) {
                const uint32_t qrow = (uint32_t)(qt * kTile + trow);
                float k1 = kWinNone, k2 = kWinNone;
                int w1 = -1, w2 = -1;
                for (int tt = 0; tt < u.ntt; ++tt, ++g) {
                    // unit = (tile, half of 64 columns); unit 2 g + half belongs to group (2 g + half) % 4: a group reads one half of every
                    // other tile, at once, and releases its share of the stage before it starts computing
                    const int half = group & 1;
                    if ((int)(g & 1u) != (group >> 1)) continue;
                    const uint32_t as = g % kWinAccStages, ab = g % kWinAccBars, aph = (g / kWinAccBars) & 1;
                    mbar_wait_sleep<kTcSleepEpilogue>(&accFull[ab], aph);
                    if (quarter == 0 && half == 0 && tt >= u.ntt - n_last) named_bar_arrive(2, 128 + 32 * n_last);
                    tc_fence_after();
                    const int c0 = tt * kTile + half * 64;
                    if constexpr (kOrb) {
                        // ---------------- ORB: 32 registers = 64 fp16 accumulators v = 256 - 2 hamming ----------------
                        uint32_t hb[32];
                        tmem_ld32_pack(tmem + lane_addr + as * 128 + half * 64, hb);
                        tmem_ld_wait();
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) mbar_arrive_relaxed(&accEmpty[ab]);
                        if (p.debug_flags & 1) continue;
                        const int rem = ft - c0;
                        if (rem < 64) {             // pad rows of the train frame (all-zero operands, only in its last tile) read as 0: mask them
#pragma unroll
                            for (int c = 0; c < 32; ++c)
                                hb[c] = 2 * c + 1 < rem ? hb[c] : (2 * c < rem ? ((hb[c] & 0xffffu) | 0xfc000000u) : 0xfc00fc00u);
                        }
                        // tournament on packed halves (even columns in the low halves, odd in the high ones), in place: sorted pairs ...
#pragma unroll
                        for (int j = 0; j < 16; ++j) {
                            const uint32_t hi = hmax2(hb[2 * j], hb[2 * j + 1]), lo = hmin2(hb[2 * j], hb[2 * j + 1]);
                            hb[2 * j] = hi; hb[2 * j + 1] = lo;
                        }
                        // ... merged down to one (largest, second) pair per 32-column part (8 pairs each): hb[0 / 1], hb[16 / 17]
#pragma unroll
                        for (int step = 1; step < 8; step <<= 1) {
#pragma unroll
                            for (int j = 0; j < 16; j += 2 * step) {
                                const uint32_t ha = hb[2 * j], la = hb[2 * j + 1], hc = hb[2 * (j + step)], lc = hb[2 * (j + step) + 1];
                                hb[2 * j] = hmax2(ha, hc);
                                hb[2 * j + 1] = hmax2(hmax2(hmin2(ha, hc), la), lc);
                            }
                        }
                        const float pm0 = fmaxf(h_lo(hb[0]), h_hi(hb[0]));
                        const uint32_t hh = hmax2(hb[0], hb[16]), ll = hmax2(hmax2(hmin2(hb[0], hb[16]), hb[1]), hb[17]);
                        const float a1 = h_lo(hh), b1 = h_hi(hh), a2 = h_lo(ll), b2 = h_hi(ll);
                        const float p1 = fmaxf(a1, b1), p2 = fmaxf(fmaxf(fminf(a1, b1), a2), b2);
                        const int sub = pm0 == p1 ? 0 : 1;                  // the lower part on ties
                        if (!(p.debug_flags & 16)) win_merge(p1, win_slice(c0 + 32 * sub, 1), p2, win_slice(c0, 2), k1, w1, k2, w2);
                    } else {
                        // ---------------- SURF: 64 fp32 accumulators v = -1/2 d^2 (pads: <= -1e30), loaded 32 at a time ----------------
                        // Chain keys: of every chain of 8 columns only its maximum is kept, and the row keeps the two largest chain maxima
                        // with their chains.  The best column lies in the best chain; the true second lies in the best chain or is the
                        // maximum of the second chain; finalize.cu evaluates the best chain exactly and so learns its own second.
                        float m[8];
#pragma unroll
                        for (int qc = 0; qc < 2; ++qc) {
                            uint32_t vb[32];
                            tmem_ld32(tmem + lane_addr + as * 128 + half * 64 + qc * 32, vb);
                            tmem_ld_wait();
                            if (qc == 1) {
                                tc_fence_before();
                                __syncwarp();
                                if (lane == 0) mbar_arrive_relaxed(&accEmpty[ab]);
                            }
#pragma unroll
                            for (int j = 0; j < 4; ++j) {
                                const float* v = reinterpret_cast<const float*>(vb) + 8 * j;
                                m[4 * qc + j] = fmaxf(fmaxf(fmaxf(v[0], v[1]), v[2]), fmaxf(fmaxf(fmaxf(v[3], v[4]), v[5]), fmaxf(v[6], v[7])));
                            }
                        }
                        if (p.debug_flags & (1 | 16)) continue;
                        // the two largest chain maxima (values: sorted pairs, merged), then the best chain, the lowest one on ties
                        const float h01 = fmaxf(m[0], m[1]), l01 = fminf(m[0], m[1]), h23 = fmaxf(m[2], m[3]), l23 = fminf(m[2], m[3]);
                        const float h45 = fmaxf(m[4], m[5]), l45 = fminf(m[4], m[5]), h67 = fmaxf(m[6], m[7]), l67 = fminf(m[6], m[7]);
                        const float ha = fmaxf(h01, h23), la = fmaxf(fmaxf(fminf(h01, h23), l01), l23);
                        const float hb = fmaxf(h45, h67), lb = fmaxf(fmaxf(fminf(h45, h67), l45), l67);
                        const float p1 = fmaxf(ha, hb), p2 = fmaxf(fmaxf(fminf(ha, hb), la), lb);
                        int j1 = 7;
#pragma unroll
                        for (int j = 6; j >= 0; --j) j1 = m[j] == p1 ? j : j1;
                        // The second chain's index is read only where both chains beat the running best (p2 > k1, win_merge): the first
                        // units of a row, rarely any later one, so it is found on a warp-uniform branch.  Lowest chain other than j1 on ties.
                        int j2 = 0;
                        if (__any_sync(0xffffffffu, p2 > k1)) {
#pragma unroll
                            for (int j = 7; j >= 0; --j) j2 = (m[j] == p2 && j != j1) ? j : j2;
                        }
                        win_merge(p1, win_slice(c0 + 8 * j1, 0), p2, win_slice(c0 + 8 * j2, 0), k1, w1, k2, w2);
                    }
                }
                // ---- end of the sweep for this query block: merge the four groups' results of every row (64-bit shared-memory atomics on
                //      packed keys, "smaller = nearer": the smallest ends in mkey[0], the smallest of all the losers in mkey[1]) ----
                const float voff = kOrb ? 256.f : 0.f;
#pragma unroll
                for (int e2 = 0; e2 < 2; ++e2) {
                    const float kv = e2 ? k2 : k1;
                    const int kw = e2 ? w2 : w1;
                    if (kw >= 0 && kv > (kOrb ? -600.f : -1.0e29f)) {          // a real column (pads: SURF <= -1e30, ORB -inf)
                        const u64 k = make_key(__float_as_uint(fmaxf(voff - kv, 0.f) + 0.f), (uint32_t)kw);   // (+ 0.f: a -0 becomes +0)
                        const u64 old = atomicMin(&mkey[trow], k);
                        atomicMin(&mkey[kTile + trow], old > k ? old : k);
                    }
                }
                asm volatile("bar.sync 1, %0;" ::"n"(kTcEpiThreads) : "memory");
                if (group == 0) {
                    if (p.gather && p.fallback) {
                        // fallback sweep: gathered row `qrow` is row gl[qrow] of the query frame (kKeyInit keeps its value under the mark)
                        if ((int)qrow < u.fq) {
                            const int r = __ldg(p.gather + (size_t)u.pair * p.stride + qrow);
                            rk1[r] = mkey[trow] | kWinExactMark;
                            rk2[r] = mkey[kTile + trow] | kWinExactMark;
                        }
                    } else if (p.gather) {
                        rk1[3 * (size_t)p.stride + qrow] = mkey[trow];      // verification sweep: the best (value, slice) of gathered row `qrow`
                    } else {
                        rk1[qrow] = mkey[trow];
                        rk2[qrow] = mkey[kTile + trow];
                    }
                    mkey[trow] = kKeyInit;
                    mkey[kTile + trow] = kKeyInit;
                }
                asm volatile("bar.sync 1, %0;" ::"n"(kTcEpiThreads) : "memory");   // mkey[] is reused by the next query block
            }
        }
    }

    // ---- teardown: everything issued has been consumed (the epilogue waited on every accumulator stage) ----
    tc_fence_before();
    __syncthreads();
    if (warp == kTcEpiWarps + 1) tmem_free(tmem, 512);
}

size_t sweep_win_smem_bytes() {
    return 1024 + (size_t)kWinStages * kWinTileBytes + kTcAugBytes + 2 * kTile * sizeof(u64) + (1 + 2 * kWinLoadBars + 2 * kWinAccBars) * 8 + 16;
}

// kind = p.tc_kind: ESFM_KIND_F32X64 (tc_main = the H images of launch_pack_tch) or ESFM_KIND_B256 (tc_main = the +-1 FP8 images)
cudaError_t launch_sweep_win(const SweepParams& p, int sm_count, cudaStream_t s) {
    const int n_units = p.n_pairs * p.units_per_pair;
    if (n_units <= 0) return cudaSuccess;
    const int grid = n_units < sm_count ? n_units : sm_count;
    const size_t smem = sweep_win_smem_bytes();
    void (*kern)(const SweepParams) = p.tc_kind == ESFM_KIND_F32X64 ? sweep_win_kernel<ESFM_KIND_F32X64> : sweep_win_kernel<ESFM_KIND_B256>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    kern<<<grid, kTcThreads, smem, s>>>(p);
    return cudaGetLastError();
}

}  // namespace esfm
