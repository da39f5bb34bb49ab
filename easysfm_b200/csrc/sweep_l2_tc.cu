// sweep_l2_tc.cu -- SURF / L2 distance sweep on the 5th-generation tensor cores (tcgen05 + TMEM), sm_100a.
//
// Same contract as sweep_l2.cu (the FP32-FFMA engine): for every image pair, the two best train rows of every
// query row and the best query row of every train row, as packed (1/2 d^2 bits << 32 | index) keys, ranked with
// OpenCV's lowest-index tie-break (BFMatcher(NORM_L2).knnMatch(k=2), python_code/feature_match.py:33-34, and the
// crossCheck of :26-27; C++ call site cpp_code/src/feature_matching.cpp:125).  finalize.cu then re-evaluates the
// candidates in direct form, so what this kernel must get right is the RANKING; its arithmetic is the 3xTF32 split
// product of tc_layout.cuh (|error| ~ 2e-6 on 1/2 d^2, measured by csrc/microbench/tc_probe.cu).
//
// The same kernel template serves ORB / Hamming (cpp_code/src/feature_matching.cpp:71-92) as an exact FP8 dot product:
// KIND = ESFM_KIND_B256 (+-1 operands, accumulator = -2 hamming, generic epilogue) and KIND = kTcKindB256Z (scaled operands
// whose accumulator is the packed key 20480 + 2^15 hamming + column: branch-free row selection; the default).
//
// One persistent CTA per SM, 24 warps, four pipelines (TMA -> shared memory -> tensor memory -> registers).  A CTA works
// on one 128-row QUERY TILE at a time and streams the train frame past it once.  (A variant with two query tiles per block,
// every train tile feeding two accumulators, measured slower in round 1 and was removed.)
//   warp 16 (one lane)  TMA producer: one cp.async.bulk per 128-row train tile image (SURF 68 KB, ORB 36 KB: main + augmented
//                       columns) into a 3-stage full/empty mbarrier ring; the 128 running column thresholds of the tile ride
//                       in their own 4-stage ring.
//   warp 17             MMA issuer (warp-uniform control flow, one elected lane issues): per train tile
//                       SURF: 25 x tcgen05.mma.cta_group::1.kind::tf32 (M=128, N=128, K=8) = 3 terms (lo.hi, hi.lo, hi.hi) x 8
//                       k-steps + 1 augmented k-step that adds both half norms exactly; ORB: 8 + 1 x kind::f8f6f4 (K=32).
//                       The query operand is read from TENSOR MEMORY, the train operand from SWIZZLE_128B shared-memory atoms;
//                       the result accumulates in one of the 3 tensor-memory stages (128 columns each);
//                       tcgen05.commit publishes the accumulator stage and releases the shared-memory stage.
//   warps 20-23         query writers: rows of the query tile -> operand columns of tensor memory (tcgen05.st; SURF: fp32 ->
//                       (hi, lo) TF32, ORB: bits -> FP8) + the tile's augmented block in shared memory; they block on a
//                       named barrier until the epilogue has seen the last accumulator that read the previous tile.
//   warps 0-15          epilogue: warp w owns TMEM lanes 32*(w%4).. (= query rows) and column quarter w/4.  tcgen05.ld
//                       gives each THREAD one query row x 32 train columns, so the row's running top-2 is thread-private
//                       (no shuffles); column minima go through a warp REDUX + one fire-and-forget atomicMin per hit.
//                       The accumulator stage is released as soon as it is in registers.
#include "tc_sweep_common.cuh"

namespace esfm {

namespace {

// Tensor memory has 512 columns: the query operand (SURF hi 64 | lo 64 = 128 columns, ORB 64) + the accumulator stages (128 columns
// each), 3 stages for both kinds.
constexpr int kTcAccStages = 3;
constexpr uint32_t kTcACol0 = 128u * kTcAccStages;     // tensor-memory column of the query operand
static_assert(kTcACol0 + 128 <= 512, "tensor memory: accumulator stages + SURF query operand");
}  // namespace

// KIND = ESFM_KIND_F32X64: 3xTF32, query operand = 128 columns (hi 64 | lo 64), train tile image 68 KB;
// KIND = ESFM_KIND_B256:   Hamming as an FP8 +-1 dot product (tc_layout.cuh), query operand = 64 columns, image 36 KB.
// KIND = kTcKindB256Z:     the same with scaled operands whose accumulator is the packed key z = Z0 + 2^15 hamming + column
//                          (tc_layout.cuh "Z" encoding): branch-free row selection.
template <int KIND>
__global__ void __launch_bounds__(kTcThreads, 1) sweep_l2_tc_kernel(const SweepParams p) {
    constexpr bool kOrb = !tc_kind_is_f32(KIND);          // FP8 operands (both ORB encodings share the MMA sequence and the tile geometry)
    constexpr bool kZ = KIND == kTcKindB256Z;
    constexpr int kTcMainBytes = kOrb ? kTc8MainBytes : esfm::kTcMainBytes;
    constexpr int kTcGroupBytes = kOrb ? kTc8GroupBytes : esfm::kTcGroupBytes;
    constexpr int kTcTileBytes = kTcMainBytes + kTcAugBytes;     // (shadows the SURF constant of tc_layout.cuh)
    constexpr uint32_t kTcBoundBits = tc_kind_is_f32(KIND) ? kTcBoundBitsF32 : (kZ ? kTcBoundBitsZ : kTcBoundBitsB256);
    extern __shared__ unsigned char smem_raw[];
    // SWIZZLE_128B atoms need 1024-byte alignment
    unsigned char* base = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    unsigned char* Ts = base;                                   // kTcStages train tile images (each 68 x 1024 B: atoms stay aligned)
    unsigned char* Qa = Ts + kTcStages * kTcTileBytes;          // augmented block (1, 1, 1, hq_h | hq_m, hq_l, 0, 0) of the query tile
    unsigned char* Thr = Qa + kTcAugBytes;                      // kTcThrStages x 128 column thresholds
    u64* mkey = reinterpret_cast<u64*>(Thr + kTcThrStages * kTcThrBytes);          // [best, second][128] merged row keys
    uint32_t* sbound = reinterpret_cast<uint32_t*>(mkey + 2 * kTile);             // [128] row bound shared by a row's parts
    float* colsc = reinterpret_cast<float*>(sbound + kTile);                      // [epilogue warp][4 columns][32 lanes] column-event scratch
    uint64_t* bars = reinterpret_cast<uint64_t*>(reinterpret_cast<unsigned char*>(colsc) + kTcScBytes);
    uint64_t* fullQ = bars;
    uint64_t* fullT = fullQ + 1;
    uint64_t* emptyT = fullT + kTcStages;
    uint64_t* accFull = emptyT + kTcStages;
    uint64_t* accEmpty = accFull + kTcAccStages;
    uint64_t* thrFull = accEmpty + kTcAccStages;
    uint64_t* thrEmpty = thrFull + kTcThrStages;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(thrEmpty + kTcThrStages);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n_units = p.n_pairs * p.units_per_pair;

    if (threadIdx.x == 0) {
        mbar_init(fullQ, 4);                          // the 4 query-writer warps
        for (int s = 0; s < kTcStages; ++s) {
            mbar_init(&fullT[s], 1);
            mbar_init(&emptyT[s], 1);                 // MMA commit
        }
        for (int s = 0; s < kTcThrStages; ++s) {
            mbar_init(&thrFull[s], 1);
            mbar_init(&thrEmpty[s], kTcEpiWarps);
        }
        for (int s = 0; s < kTcAccStages; ++s) {
            mbar_init(&accFull[s], 1);
            mbar_init(&accEmpty[s], kTcEpiWarps);
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
                const TcUnit u = tc_decode_unit(p, unit);
                const unsigned char* timg = p.tc_main + (size_t)p.frame_tile_off[u.t_frame] * kTcTileBytes;
                const uint32_t* tauc = p.col_thr + (size_t)u.pair * p.stride;
                for (int qt = u.qb0; qt < u.qb1; ++qt) {
                    for (int tt = 0; tt < u.ntt; ++tt, ++g) {
                        const uint32_t st = g % kTcStages, ph = (g / kTcStages) & 1;
                        mbar_wait_sleep<kTcSleepProducer>(&emptyT[st], ph ^ 1);
                        mbar_arrive_expect_tx(&fullT[st], kTcTileBytes);
                        if (p.debug_flags & 4)
                            asm volatile("mbarrier.complete_tx.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(&fullT[st])), "r"(kTcTileBytes) : "memory");
                        else
                            bulk_g2s(Ts + (size_t)st * kTcTileBytes, timg + (size_t)tt * kTcTileBytes, kTcTileBytes, &fullT[st]);
                        // the running column thresholds of this tile ride along in their own ring (a snapshot a few tiles
                        // old is fine: a stale threshold is only looser, never wrong)
                        const uint32_t ts = g % kTcThrStages, tph = (g / kTcThrStages) & 1;
                        mbar_wait_sleep<kTcSleepProducer>(&thrEmpty[ts], tph ^ 1);
                        mbar_arrive_expect_tx(&thrFull[ts], kTcThrBytes);
                        bulk_g2s(Thr + ts * kTcThrBytes, tauc + (size_t)tt * kTile, kTcThrBytes, &thrFull[ts]);
                    }
                }
            }
        }
    } else if (warp == kTcEpiWarps + 1) {
        // ======================= MMA issuer =======================
        // The WHOLE warp walks the loops and waits on the barriers (warp-uniform control flow, so the shared-memory
        // descriptors live in uniform registers); one elected lane issues the tcgen05.mma / tcgen05.commit instructions.
        // (Issuing from inside `if (lane == 0)` made the compiler wrap every MMA in an ELECT / R2UR.BROADCAST waterfall
        // loop: 16 dependent instructions and ~90 cycles per MMA, longer than the MMA itself.)
        constexpr uint32_t idesc = kOrb ? tc_idesc_e4m3(128, 128) : tc_idesc_tf32(128, 128);
        const uint64_t qad0 = tc_desc_nosw(smem_u32(Qa), 128, kTcAugGroupBytes);
        const uint64_t td0 = tc_desc_sw128(smem_u32(Ts), kTcGroupBytes);
        const uint64_t tad0 = tc_desc_nosw(smem_u32(Ts) + kTcMainBytes, 128, kTcAugGroupBytes);
        const uint32_t acol = tmem + kTcACol0;
        uint32_t g = 0;                      // train tiles streamed = accumulator jobs issued
        uint32_t qn = 0;                     // how many times the query operand has been filled
        for (int unit = blockIdx.x; unit < n_units; unit += gridDim.x) {
            const TcUnit u = tc_decode_unit(p, unit);
            for (int qt = u.qb0; qt < u.qb1; ++qt, ++qn) {
                for (int tt = 0; tt < u.ntt; ++tt, ++g) {
                    const uint32_t st = g % kTcStages, ph = (g / kTcStages) & 1;
                    mbar_wait_sleep<kTcSleepIssuer>(&fullT[st], ph);
                    // descriptor start addresses are in 16-byte units: adding (bytes >> 4) to the low word moves the window
                    const uint64_t td = td0 + (uint64_t)(st * (kTcTileBytes >> 4));
                    const uint64_t tad = tad0 + (uint64_t)(st * (kTcTileBytes >> 4));
                    const uint32_t as = g % kTcAccStages, aph = (g / kTcAccStages) & 1;
                    if (tt == 0) mbar_wait_sleep<kTcSleepIssuer>(fullQ, qn & 1);   // the writers have filled the query operand for this tile
                    mbar_wait_sleep<kTcSleepIssuer>(&accEmpty[as], aph ^ 1);
                    tc_fence_after();
                    const uint32_t d = tmem + as * 128;
                    if (kOrb) {
                        if (!(p.debug_flags & 2) && elect_one()) {
                            // 256 FP8 values per row = 8 k-steps of K = 32 (32 bytes: the same descriptor arithmetic as TF32's K = 8)
#pragma unroll
                            for (int ks = 0; ks < 8; ++ks) {
                                const uint32_t off = ((ks >> 2) * 1024 + (ks & 3) * 32) >> 4;
                                tc_mma_f8_ts(d, acol + ks * 8, td + (uint64_t)off, idesc, ks > 0);
                            }
                            // - 256 and the pad-row penalties (tc_layout.cuh)
                            tc_mma_f8(d, qad0, tad, idesc, true);
                        }
                    } else
                    if (!(p.debug_flags & 2) && elect_one()) {
                        bool first = true;
#pragma unroll
                        for (int term = 0; term < 3; ++term) {
                            // (A part, B part): lo.hi, hi.lo first (small terms), hi.hi last
                            const int pa = term == 0 ? 1 : 0, pb = term == 1 ? 1 : 0;
#pragma unroll
                            for (int ks = 0; ks < 8; ++ks) {
                                const uint32_t off = ((ks >> 2) * 1024 + (ks & 3) * 32) >> 4;
                                // A (query) from tensor memory: lane = row, column = k.  With both operands in shared memory the
                                // 8 KB of operand reads per MMA plus the TMA writes saturate the 128 B/clk shared-memory port
                                // (measured 87 cycles per MMA instead of 64).
                                tc_mma_tf32_ts(d, acol + pa * 64 + ks * 8, td + (uint64_t)(pb * (2048 >> 4) + off), idesc, !first);
                                first = false;
                            }
                        }
                        // - 1/2|q|^2 - 1/2|t|^2, exact (three-way split half norms against ones)
                        tc_mma_tf32(d, qad0, tad, idesc, true);
                    }
                    __syncwarp();
                    if (elect_one()) {
                        tc_commit(&accFull[as]);                        // accumulator stage ready for the epilogue
                        tc_commit(&emptyT[st]);                         // shared-memory stage consumed
                    }
                    __syncwarp();
                }
            }
        }
    } else if (warp >= kTcWriterWarp0) {
        // ======================= query writers: fp32 rows -> (hi, lo) TF32 operand in tensor memory =======================
        const int quarter = warp & 3;
        const int trow = quarter * 32 + lane;
        const uint32_t lane_addr = (uint32_t)(quarter * 32) << 16;
        bool filled = false;                // the query operand has been filled before: wait until the epilogue is done with it
        for (int unit = blockIdx.x; unit < n_units; unit += gridDim.x) {
            const TcUnit u = tc_decode_unit(p, unit);
            const int fq = p.frame_rows[u.q_frame];
            if (kOrb) {
                // ---- ORB: 256 bits -> 256 FP8 values +-1.0 (Z encoding: +-256), 4 per tensor-memory column ----
                const uint4* qbits = p.rows_b256 + (size_t)p.frame_row_off[u.q_frame] * 2;
                for (int qt = u.qb0; qt < u.qb1; ++qt) {
                    const int r = qt * kTile + trow;
                    const bool valid = r < fq;
                    uint4 w0 = make_uint4(0u, 0u, 0u, 0u), w1 = w0;
                    if (valid) { w0 = __ldg(qbits + (size_t)r * 2); w1 = __ldg(qbits + (size_t)r * 2 + 1); }
                    if (filled) named_bar_sync(2, 128 + 32);      // operand free (see the SURF branch below)
                    filled = true;
                    tc_fence_after();
                    // augmented columns: (qpad ? 448 : 0, 448, 16, 0 ...) in FP8; Z encoding: the offset slots and digit multipliers
                    unsigned char* qa = Qa + (trow >> 3) * kTcAugGroupBytes + (trow & 7) * 16;
                    if (kZ) {
                        uint32_t aw[8];
                        tcz_query_aug(aw);
                        *reinterpret_cast<uint4*>(qa) = make_uint4(aw[0], aw[1], aw[2], aw[3]);
                        *reinterpret_cast<uint4*>(qa + 128) = make_uint4(aw[4], aw[5], aw[6], aw[7]);
                    } else {
                        *reinterpret_cast<uint4*>(qa) = make_uint4((valid ? 0u : kFp8Pos448) | (kFp8Pos448 << 8) | (kFp8Pos16 << 16), 0u, 0u, 0u);
                        *reinterpret_cast<uint4*>(qa + 128) = make_uint4(0u, 0u, 0u, 0u);
                    }
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                    const uint32_t acol = tmem + lane_addr + kTcACol0;
                    const uint32_t ws[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
#pragma unroll
                    for (int m = 0; m < 8; ++m) {       // word m = elements 32 m .. 32 m + 31 = 8 columns
                        uint32_t c[8];
#pragma unroll
                        for (int j = 0; j < 8; ++j) c[j] = valid ? (kZ ? tcz_expand4_q(ws[m] >> (4 * j)) : tc8_expand4(ws[m] >> (4 * j))) : 0u;
                        tmem_st8(acol + m * 8, c);
                    }
                    tmem_st_wait();
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(fullQ);
                }
                continue;
            }
            const float4* qrows = reinterpret_cast<const float4*>(p.rows_f32 + (size_t)p.frame_row_off[u.q_frame] * kDim);
            for (int qt = u.qb0; qt < u.qb1; ++qt) {
                const int r = qt * kTile + trow;
                const bool valid = r < fq;
                const float4* xr = qrows + (size_t)(valid ? r : 0) * 16;
                // pass 1: 1/2|q|^2 in the summation order of bank.cu's pack kernels (few live registers: this warpgroup runs at 40)
                float hs = 0.f;
#pragma unroll 4
                for (int m = 0; m < 16; ++m) {
                    const float4 x = __ldg(xr + m);
                    hs = __fmaf_rn(x.x, x.x, hs); hs = __fmaf_rn(x.y, x.y, hs);
                    hs = __fmaf_rn(x.z, x.z, hs); hs = __fmaf_rn(x.w, x.w, hs);
                }
                float hq = valid ? 0.5f * hs : kTcPadNorm;   // pad rows can never win a column
                float hqh, hqm, hql;
                tc_split3(hq, hqh, hqm, hql);
                // The operand is free once every MMA that read the previous query tile has retired.  The writers do not poll for
                // that (four warps polling an mbarrier for a whole query tile were 20 % of all executed instructions; __nanosleep does
                // not sleep anywhere near the requested time): they block on NAMED BARRIER 2, which epilogue warp 0 arrives at as
                // soon as it has seen the accumulator of the previous tile's last train tile complete.
                if (filled) named_bar_sync(2, 128 + 32);
                filled = true;
                tc_fence_after();
                unsigned char* qa = Qa + (trow >> 3) * kTcAugGroupBytes + (trow & 7) * 16;
                *reinterpret_cast<float4*>(qa) = make_float4(1.f, 1.f, 1.f, hqh);
                *reinterpret_cast<float4*>(qa + 128) = make_float4(hqm, hql, 0.f, 0.f);
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy stores -> visible to the MMA's async reads
                const uint32_t acol = tmem + lane_addr + kTcACol0;
                // pass 2: the row again (L1/L2 hit), 8 dims at a time -> hi / lo columns of tensor memory
#pragma unroll 2
                for (int m = 0; m < 8; ++m) {
                    float4 x0 = __ldg(xr + 2 * m), x1 = __ldg(xr + 2 * m + 1);
                    if (!valid) { x0 = make_float4(0.f, 0.f, 0.f, 0.f); x1 = x0; }
                    const float xs[8] = {x0.x, x0.y, x0.z, x0.w, x1.x, x1.y, x1.z, x1.w};
                    uint32_t hi[8], lo[8];
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const float hv = tc_tf32_hi(xs[j]);
                        hi[j] = __float_as_uint(hv);
                        lo[j] = __float_as_uint(xs[j] - hv);
                    }
                    tmem_st8(acol + m * 8, hi);
                    tmem_st8(acol + 64 + m * 8, lo);
                }
                tmem_st_wait();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(fullQ);
            }
        }
        // the epilogue arrives once per query tile; the last arrival has no refill waiting for it
        if (filled) named_bar_sync(2, 128 + 32);
    }
    } else {
        // ======================= epilogue warps =======================
        reg_alloc<kTcEpiRegs>();
        const int quarter = warp & 3, part = warp >> 2;
        const int trow = quarter * 32 + lane;               // row inside a 128-row query tile (= TMEM lane)
        const uint32_t lane_addr = (uint32_t)(quarter * 32) << 16;
        if (part == 0) {
            sbound[trow] = kTcBoundBits;
            mkey[trow] = kKeyInit;
            mkey[kTile + trow] = kKeyInit;
        }
        asm volatile("bar.sync 1, %0;" ::"n"(kTcEpiThreads) : "memory");
        uint32_t g = 0;                     // train tiles seen = accumulators read
        for (int unit = blockIdx.x; unit < n_units; unit += gridDim.x) {
            const TcUnit u = tc_decode_unit(p, unit);
            u64* rk1 = p.keys + (size_t)u.pair * 4 * p.stride;
            u64* rk2 = rk1 + p.stride;
            u64* ck1 = rk2 + p.stride;
            uint32_t* tauc = p.col_thr + (size_t)u.pair * p.stride;
            for (int qt = u.qb0; qt < u.qb1; ++qt) {
                if constexpr (kZ) {
                    // ================= ORB, "Z" encoding: the accumulator IS the packed key z = Z0 + 2^15 hamming + column =================
                    // Every element of a row is a distinct positive integer-valued float, smaller = nearer, ties = lower column, so the
                    // row's two nearest neighbours are the two smallest values this thread ever reads: three FMNMX per element, no
                    // bound, no slow path, no tie logic.  Columns keep the threshold scheme (their minimum runs over other warps' rows).
                    const int fq = p.frame_rows[u.q_frame], ft = p.frame_rows[u.t_frame];
                    const uint32_t qrow = (uint32_t)(qt * kTile + trow);
                    const bool qvalid = (int)qrow < fq;          // pad query rows read as z = Z0 + 2^22 + column: they must not win a column
                    // One CTA per pair (units_per_pair == 1): a threshold snapshot only ever holds minima of LOWER query rows (earlier
                    // query blocks; this block's own updates come after the snapshot was taken), so an equal distance can never win and
                    // the published threshold may exclude it (z - 1: same column, same distance => same z).  With the pair split over
                    // several CTAs other CTAs' (higher) rows are in the snapshot too and equal distances must still get through.
                    const float thr_sub = p.units_per_pair == 1 ? 1.f : 0.f;
                    float k1 = kTcZNone, k2 = kTcZNone;
                    for (int tt = 0; tt < u.ntt; ++tt, ++g) {
                        const uint32_t ts = g % kTcThrStages, tph = (g / kTcThrStages) & 1;
                        mbar_wait_sleep<kTcSleepEpilogue>(&thrFull[ts], tph);
                        const float4* tp = reinterpret_cast<const float4*>(Thr + ts * kTcThrBytes) + part * (kTcPartCols / 4);
                        const uint32_t as = g % kTcAccStages, aph = (g / kTcAccStages) & 1;
                        mbar_wait_sleep<kTcSleepEpilogue>(&accFull[as], aph);
                        if (warp == 0 && tt == u.ntt - 1) named_bar_arrive(2, 128 + 32);     // the query operand may be refilled (see the writers)
                        tc_fence_after();
                        uint32_t vb[32];
                        tmem_ld32(tmem + lane_addr + as * 128 + part * kTcPartCols, vb);
                        tmem_ld_wait();
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) mbar_arrive_relaxed(&accEmpty[as]);
                        if (!(p.debug_flags & 1)) {
                            const uint32_t col0 = (uint32_t)(tt * kTile + part * kTcPartCols);
                            if (tt == u.ntt - 1) {       // only the last tile of a frame has pad rows (all-zero operands: z = 0)
                                // masked IN PLACE (predicated moves): a select into new registers made the compiler copy all 32
                                // accumulators on every pass of every tile
    #pragma unroll
                                for (int c = 0; c < 32; ++c)
                                    asm volatile("{\n\t.reg .pred p;\n\tsetp.ge.s32 p, %1, %2;\n\t@p mov.b32 %0, 0x7f61b1e6;\n\t}"      // kTcZNone = 3.0e38f
                                                 : "+r"(vb[c]) : "r"((int)(col0 + c)), "r"(ft));
                            }
                            float v[32];
    #pragma unroll
                            for (int c = 0; c < 32; ++c) v[c] = __uint_as_float(vb[c]);
                            // ---- rows: running two smallest ----
                            if (!(p.debug_flags & 16)) {
    #pragma unroll
                            for (int c = 0; c < 32; ++c) {
                                const float hi = fmaxf(k1, v[c]);
                                k1 = fminf(k1, v[c]);
                                k2 = fminf(k2, hi);
                            }
                            }
                            // ---- columns: 4 chains of 8 threshold tests, one vote ----
                            if (p.need_cols) {
                            bool cf[4];
    #pragma unroll
                            for (int cq = 0; cq < 4; ++cq) {
                                const float4 x0 = tp[2 * cq], x1 = tp[2 * cq + 1];
                                cf[cq] = qvalid & ((v[8 * cq] <= x0.x) | (v[8 * cq + 1] <= x0.y) | (v[8 * cq + 2] <= x0.z) | (v[8 * cq + 3] <= x0.w) |
                                                   (v[8 * cq + 4] <= x1.x) | (v[8 * cq + 5] <= x1.y) | (v[8 * cq + 6] <= x1.z) | (v[8 * cq + 7] <= x1.w));
                            }
                            if (!(p.debug_flags & 8) && __any_sync(0xffffffffu, cf[0] | cf[1] | cf[2] | cf[3])) {
                                // Column events: ~0.7 per pass, plus 32 per pass in the first query block of a pair (every column gets its
                                // first minimum there: 60 % of all events).  Per group of 4 columns with a hit: park the group in the
                                // warp's scratch, then ONE segmented warp reduction over its four columns (tc_col_group).
                                const uint32_t sc_addr = smem_u32(colsc) + (uint32_t)warp * (kTcScCols * 32 * 4);
                                const uint32_t thr_addr = smem_u32(tp);
                                u64* ckb = ck1 + col0;
                                uint32_t* taub = tauc + col0;
                                asm volatile("" : "+l"(ckb), "+l"(taub));          // computed once per pass, not once per group
                                const uint32_t qrow0 = (uint32_t)(qt * kTile + quarter * 32);
    #pragma unroll
                                for (int cq = 0; cq < 4; ++cq) {
                                    const uint32_t hm = __ballot_sync(0xffffffffu, cf[cq]);
                                    if (hm == 0) continue;
                                    if (__popc(hm) <= 4) {
                                        // few rows beat this chain's thresholds (the steady state): each posts its own keys, straight-line
                                        const float4 x0 = tp[2 * cq], x1 = tp[2 * cq + 1];
                                        u64* ckc = ckb + 8 * cq;
                                        uint32_t* tac = taub + 8 * cq;
                                        tc_col_post<0>(v[8 * cq], x0.x, qvalid, ckc, tac, qrow, thr_sub);
                                        tc_col_post<1>(v[8 * cq + 1], x0.y, qvalid, ckc, tac, qrow, thr_sub);
                                        tc_col_post<2>(v[8 * cq + 2], x0.z, qvalid, ckc, tac, qrow, thr_sub);
                                        tc_col_post<3>(v[8 * cq + 3], x0.w, qvalid, ckc, tac, qrow, thr_sub);
                                        tc_col_post<4>(v[8 * cq + 4], x1.x, qvalid, ckc, tac, qrow, thr_sub);
                                        tc_col_post<5>(v[8 * cq + 5], x1.y, qvalid, ckc, tac, qrow, thr_sub);
                                        tc_col_post<6>(v[8 * cq + 6], x1.z, qvalid, ckc, tac, qrow, thr_sub);
                                        tc_col_post<7>(v[8 * cq + 7], x1.w, qvalid, ckc, tac, qrow, thr_sub);
                                        continue;
                                    }
                                    // many rows at once (the first query block of a pair: no bounds yet): one winner per column and warp
    #pragma unroll
                                    for (int g2 = 0; g2 < 2; ++g2) {
                                        const int gq = 2 * cq + g2;
    #pragma unroll
                                        for (int e = 0; e < 4; ++e)     // pad query rows (z = Z0 + 2^22 + column) must never win a column
                                            asm volatile("st.shared.f32 [%0], %1;" ::"r"(sc_addr + (uint32_t)(e * 128) + (uint32_t)lane * 4u), "f"(qvalid ? v[4 * gq + e] : kTcZNone) : "memory");
                                        __syncwarp();
                                        if (!(p.debug_flags & 64)) tc_col_group<true>(sc_addr, thr_addr + 16u * gq, ckb + 4 * gq, taub + 4 * gq, qrow0, thr_sub, p.debug_flags);
                                        __syncwarp();
                                    }
                                }
                            }
                            }
                        }
                        __syncwarp();
                        if (lane == 0) mbar_arrive_relaxed(&thrEmpty[ts]);      // last read of this threshold snapshot
                    }
                    // merge the four column parts of the row: two smallest keys of (up to) eight; the column comes out of the key
    #pragma unroll
                    for (int e = 0; e < 2; ++e) {
                        const float z = e ? k2 : k1;
                        if (z < 1.6e7f) {
                            const uint32_t idx = (uint32_t)((int)z - kTcZ0i) & (uint32_t)(kTcZMaxRows - 1);
                            const u64 k = make_key(__float_as_uint(z), idx);
                            const u64 old = atomicMin(&mkey[trow], k);
                            atomicMin(&mkey[kTile + trow], old > k ? old : k);
                        }
                    }
                } else {
                    // running top-2 of this thread's row
                    RowTop2 t;
                    t.v1 = t.v2 = __uint_as_float(kTcBoundBits);
                    t.i1 = t.i2 = 0xffffffffu;
                    const uint32_t qrow = (uint32_t)(qt * kTile + trow);     // frame row of this thread
                    uint32_t* sb = &sbound[trow];
                    for (int tt = 0; tt < u.ntt; ++tt, ++g) {
                        const uint32_t ts = g % kTcThrStages, tph = (g / kTcThrStages) & 1;
                        mbar_wait_sleep<kTcSleepEpilogue>(&thrFull[ts], tph);
                        const float4* tp = reinterpret_cast<const float4*>(Thr + ts * kTcThrBytes) + part * (kTcPartCols / 4);
                        const uint32_t as = g % kTcAccStages, aph = (g / kTcAccStages) & 1;
                        mbar_wait_sleep<kTcSleepEpilogue>(&accFull[as], aph);
                        if (warp == 0 && tt == u.ntt - 1) named_bar_arrive(2, 128 + 32);   // the query operand may be refilled (see the writers)
                        tc_fence_after();
                        // All 32 columns of this thread go to registers at once and the accumulator stage is released right
                        // away: the tensor pipe never waits for the selection logic below.
                        uint32_t vb[32];
                        tmem_ld32(tmem + lane_addr + as * 128 + part * kTcPartCols, vb);
                        // The row's running second best over ALL column parts (each part keeps a private top-2; the shared
                        // bound only filters, with '>=' so equal values still reach the private strict-'<' insertion).
                        float nb = -__uint_as_float(*reinterpret_cast<volatile uint32_t*>(sb));
                        tmem_ld_wait();
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) mbar_arrive_relaxed(&accEmpty[as]);
                        if (!(p.debug_flags & 1)) {
                            float v[32];
    #pragma unroll
                            for (int c = 0; c < 32; ++c) v[c] = __uint_as_float(vb[c]);   // v = -1/2 d^2
                            // ---- fast path: maxima of 8 groups of 4 columns -> one row test; 4 chains of 8 column tests; ONE vote ----
                            float gm[8];
    #pragma unroll
                            for (int gq = 0; gq < 8; ++gq)
                                gm[gq] = fmaxf(fmaxf(fmaxf(v[4 * gq], v[4 * gq + 1]), v[4 * gq + 2]), v[4 * gq + 3]);
                            const float rmax = fmaxf(fmaxf(fmaxf(fmaxf(gm[0], gm[1]), gm[2]), fmaxf(fmaxf(gm[3], gm[4]), gm[5])), fmaxf(gm[6], gm[7]));
                            const bool rflag = rmax >= nb && !(p.debug_flags & 16);
                            // (A pre-test on one threshold per group of 4 columns -- 8 compares and 2 loads instead of 32 and 8 -- was
                            // tried and lost 15 %: the loosest of four thresholds lets far too many rows through to the slow path.)
                            bool cf[4] = {false, false, false, false};
                            if (p.need_cols) {
    #pragma unroll
                                for (int cq = 0; cq < 4; ++cq) {
                                    const float4 x0 = tp[2 * cq], x1 = tp[2 * cq + 1];
                                    cf[cq] = (v[8 * cq] >= -x0.x) | (v[8 * cq + 1] >= -x0.y) | (v[8 * cq + 2] >= -x0.z) | (v[8 * cq + 3] >= -x0.w) |
                                             (v[8 * cq + 4] >= -x1.x) | (v[8 * cq + 5] >= -x1.y) | (v[8 * cq + 6] >= -x1.z) | (v[8 * cq + 7] >= -x1.w);
                                }
                            }
                            const bool cflag = (cf[0] | cf[1] | cf[2] | cf[3]) && !(p.debug_flags & 8);
                            if (__any_sync(0xffffffffu, rflag || cflag)) {
                                // ---- slow path: ~2 ln F hits per row and ~ln F per column over a whole sweep ----
                                const uint32_t col0 = (uint32_t)(tt * kTile + part * kTcPartCols);
                                // columns first (the row insertion below retires elements of v[])
                                if (__any_sync(0xffffffffu, cflag)) {
                                    // per group of 4 columns with a hit: park the group in the warp's scratch, then the compact shared
                                    // segmented warp reduction (tc_col_group; ~0.5 events per pass + 32 per pass in the first query block of a pair)
                                    const uint32_t sc_addr = smem_u32(colsc) + (uint32_t)warp * (kTcScCols * 32 * 4);
                                    const uint32_t thr_addr = smem_u32(tp);
                                    u64* ckb = ck1 + col0;
                                    uint32_t* taub = tauc + col0;
                                    asm volatile("" : "+l"(ckb), "+l"(taub));      // computed once per pass, not once per group
                                    const uint32_t qrow0 = qrow - (uint32_t)lane;
    #pragma unroll
                                    for (int cq = 0; cq < 4; ++cq) {
                                        const uint32_t hm = __ballot_sync(0xffffffffu, cf[cq] && cflag);
                                        if (hm == 0) continue;
                                        if (__popc(hm) <= 4) {
                                            // few rows beat this chain's thresholds (the steady state): each posts its own keys, straight-line
                                            const float4 x0 = tp[2 * cq], x1 = tp[2 * cq + 1];
                                            u64* ckc = ckb + 8 * cq;
                                            uint32_t* tac = taub + 8 * cq;
                                            tc_col_post<0>(fmaxf(-v[8 * cq], 0.f), x0.x, 1, ckc, tac, qrow, 0.f);
                                            tc_col_post<1>(fmaxf(-v[8 * cq + 1], 0.f), x0.y, 1, ckc, tac, qrow, 0.f);
                                            tc_col_post<2>(fmaxf(-v[8 * cq + 2], 0.f), x0.z, 1, ckc, tac, qrow, 0.f);
                                            tc_col_post<3>(fmaxf(-v[8 * cq + 3], 0.f), x0.w, 1, ckc, tac, qrow, 0.f);
                                            tc_col_post<4>(fmaxf(-v[8 * cq + 4], 0.f), x1.x, 1, ckc, tac, qrow, 0.f);
                                            tc_col_post<5>(fmaxf(-v[8 * cq + 5], 0.f), x1.y, 1, ckc, tac, qrow, 0.f);
                                            tc_col_post<6>(fmaxf(-v[8 * cq + 6], 0.f), x1.z, 1, ckc, tac, qrow, 0.f);
                                            tc_col_post<7>(fmaxf(-v[8 * cq + 7], 0.f), x1.w, 1, ckc, tac, qrow, 0.f);
                                            continue;
                                        }
                                        // many rows at once (the first query block of a pair: no bounds yet): one winner per column and warp
    #pragma unroll
                                        for (int g2 = 0; g2 < 2; ++g2) {
                                            const int gq = 2 * cq + g2;
    #pragma unroll
                                            for (int e = 0; e < 4; ++e)     // keys: 1/2 d^2 clamped at 0 (pad query rows: 1e30, never a winner)
                                                asm volatile("st.shared.f32 [%0], %1;" ::"r"(sc_addr + (uint32_t)(e * 128) + (uint32_t)lane * 4u), "f"(fmaxf(-v[4 * gq + e], 0.f)) : "memory");
                                            __syncwarp();
                                            if (!(p.debug_flags & 64)) tc_col_group<false>(sc_addr, thr_addr + 16u * gq, ckb + 4 * gq, taub + 4 * gq, qrow0, 0.f, p.debug_flags);
                                            __syncwarp();
                                        }
                                    }
                                }
                                if (rflag) {
                                    // Per group of 4 columns a LOOP (a real branch, never if-converted) that takes the group's maximum while it
                                    // still beats the bound: insert it, retire it, recompute the group maximum.  Typically one trip in
                                    // one group.  Equal values leave the group lowest column first, so ascending-index ties hold.
                                    bool ins = false;
    #pragma unroll
                                    for (int gq = 0; gq < 8; ++gq) {
                                        while (gm[gq] >= nb) {
                                            const float m = gm[gq], d = -m;
                                            if (!(d < t.v2)) break;     // let through by another part's bound or an equal value: nothing here can enter
                                            const int j = v[4 * gq] == m ? 0 : (v[4 * gq + 1] == m ? 1 : (v[4 * gq + 2] == m ? 2 : 3));
                                            const uint32_t idx = col0 + 4 * gq + j;
                                            if (d < t.v1) {
                                                t.v2 = t.v1; t.i2 = t.i1;
                                                t.v1 = d;    t.i1 = idx;
                                            } else {
                                                t.v2 = d;    t.i2 = idx;
                                            }
                                            ins = true;
                                            nb = fmaxf(nb, -t.v2);
    #pragma unroll
                                            for (int e = 0; e < 4; ++e) v[4 * gq + e] = (e == j) ? -3.0e38f : v[4 * gq + e];
                                            gm[gq] = fmaxf(fmaxf(fmaxf(v[4 * gq], v[4 * gq + 1]), v[4 * gq + 2]), v[4 * gq + 3]);
                                        }
                                    }
                                    if (ins) atomicMin(sb, __float_as_uint(fmaxf(t.v2, 0.f)));
                                }
                            }
                        }
                        __syncwarp();
                        if (lane == 0) mbar_arrive_relaxed(&thrEmpty[ts]);      // last read of this threshold snapshot
                    }
                    // ---- end of the sweep for this query block: merge the column parts of every row, publish ----
                    // 64-bit shared-memory atomics on packed keys: the smallest key ends in mkey[0][.], the smallest of all the
                    // "losers" (displaced old minimum, or the newcomer if it did not win) in mkey[1][.] = the second smallest overall.
    #pragma unroll
                    for (int e = 0; e < 2; ++e) {
                        const uint32_t idx = e ? t.i2 : t.i1;
                        if (idx != 0xffffffffu) {
                            const u64 k = make_key(__float_as_uint(fmaxf(e ? t.v2 : t.v1, 0.f)), idx);
                            const u64 old = atomicMin(&mkey[trow], k);
                            atomicMin(&mkey[kTile + trow], old > k ? old : k);
                        }
                    }
                }   // (generic epilogue)
                asm volatile("bar.sync 1, %0;" ::"n"(kTcEpiThreads) : "memory");
                if (part == 0) {       // column part 0 publishes (and resets) the query tile
                    const uint32_t qrow = (uint32_t)(qt * kTile + trow);
                    rk1[qrow] = mkey[trow];
                    rk2[qrow] = mkey[kTile + trow];
                    mkey[trow] = kKeyInit;
                    mkey[kTile + trow] = kKeyInit;
                    sbound[trow] = kTcBoundBits;
                }
                asm volatile("bar.sync 1, %0;" ::"n"(kTcEpiThreads) : "memory");   // mkey[] / sbound[] are reused by the next query block
            }
        }
    }

    // ---- teardown: everything issued has been consumed (the epilogue waited on every accumulator stage) ----
    tc_fence_before();
    __syncthreads();
    if (warp == kTcEpiWarps + 1) tmem_free(tmem, 512);
}

size_t sweep_tc_smem_bytes(int kind) {
    const size_t tile = tc_kind_is_f32(kind) ? (size_t)kTcTileBytes : (size_t)kTc8TileBytes;
    return 1024 + (size_t)kTcStages * tile + (size_t)kTcAugBytes + (size_t)kTcThrStages * kTcThrBytes +
           (size_t)2 * kTile * sizeof(u64) + (size_t)kTile * 4 + (size_t)kTcScBytes +
           (1 + 2 * kTcStages + 2 * kTcAccStages + 2 * kTcThrStages) * 8 + 16;
}

// kind = p.tc_kind: ESFM_KIND_F32X64 (3xTF32 L2 sweep) or ESFM_KIND_B256 (FP8 Hamming sweep)
cudaError_t launch_sweep_l2_tc(const SweepParams& p, int sm_count, cudaStream_t s) {
    const int n_units = p.n_pairs * p.units_per_pair;
    if (n_units <= 0) return cudaSuccess;
    const int grid = n_units < sm_count ? n_units : sm_count;
    const int kind = p.tc_kind == kTcKindB256Z ? p.tc_kind : (p.tc_kind == ESFM_KIND_B256 ? ESFM_KIND_B256 : ESFM_KIND_F32X64);
    const size_t smem = sweep_tc_smem_bytes(kind);
    void (*kern)(const SweepParams) =
        kind == kTcKindB256Z ? sweep_l2_tc_kernel<kTcKindB256Z>
        : kind == ESFM_KIND_B256 ? sweep_l2_tc_kernel<ESFM_KIND_B256> : sweep_l2_tc_kernel<ESFM_KIND_F32X64>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    kern<<<grid, kTcThreads, smem, s>>>(p);
    return cudaGetLastError();
}

}  // namespace esfm
