// sweep_l2.cu -- SURF / L2 distance sweep for sm_100a: the FP32-pipe hot kernel.
//
// Replaces the Fq x Ft x 64 distance loop + per-row top-K insertion inside OpenCV's
// BFMatcher::knnMatchImpl -> cv::batchDistance that the reference reaches from
// python_code/feature_match.py:33-34 (BFMatcher(NORM_L2).knnMatch(k=2)) and, for the cross-check,
// feature_match.py:26-27; the C++ twin of the call site is cpp_code/src/feature_matching.cpp:125.
//
// One persistent CTA per SM walks work units (image pair x range of 256-row query blocks):
//   producer warp : one elected lane streams k-major 128-row tiles (33,280 B each: 64x128 operands +
//                   128 half squared norms) global -> shared with cp.async.bulk (TMA, UBLKCP) through a
//                   STAGES-deep full/empty mbarrier ring; the 256-row query block has its own barrier pair.
//   8 consumer warps : each thread owns an 8-row x 16-column register tile of
//                   acc = 1/2|q|^2 + 1/2|t|^2 - q.t  (= 1/2 d^2, exact FP32 FMAs, issued as packed FFMA2
//                   so the FMA pipe saturates at half the issue slots; operands via LDS.128, 6 per k-step).
//   epilogue      : acc <= threshold compares against the running second-best of the row (shared memory,
//                   per query block) and of the column (shared memory, per pair).  Hits are rare
//                   (~2 ln F per row/column); they go through 64-bit atomicMin on packed
//                   (distance bits << 32 | index) keys, whose unsigned order is (distance, lowest index) --
//                   OpenCV's tie-break.  The distance matrix never leaves registers.
// The keys hold the two best candidates per query row AND per train row (for the mutual cross-check);
// finalize.cu re-evaluates them in direct form sum (a-b)^2 (SURVEY.md F10) before the ratio test.
#include "esfm_internal.cuh"

namespace esfm {

namespace {

__device__ __forceinline__ float4 lds128(const float* p) { return *reinterpret_cast<const float4*>(p); }

__device__ __forceinline__ uint4 ldcg_u4(const uint32_t* p) {   // L2-coherent 128-bit load (other CTAs update these)
    uint4 v;
    asm volatile("ld.global.cg.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
    return v;
}

__device__ __forceinline__ uint4 lds128_volatile_u32(const uint32_t* p) {
    uint4 v;
    asm volatile("ld.volatile.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(smem_u32(p)));
    return v;
}

struct UnitInfo {
    int pair, q_frame, t_frame;
    int nqt, ntt;      // tiles in query / train frame
    int qb0, qb1;      // query-block range of this unit
};

__device__ __forceinline__ UnitInfo decode_unit(const SweepParams& p, int unit) {
    UnitInfo u;
    u.pair = unit / p.units_per_pair;
    const int part = unit - u.pair * p.units_per_pair;
    const PairDesc pd = p.pairs[u.pair];
    u.q_frame = pd.q_frame;
    u.t_frame = pd.t_frame;
    u.nqt = p.frame_tile_off[pd.q_frame + 1] - p.frame_tile_off[pd.q_frame];
    u.ntt = p.frame_tile_off[pd.t_frame + 1] - p.frame_tile_off[pd.t_frame];
    const int nqb = (u.nqt + kQTiles - 1) / kQTiles;
    u.qb0 = (int)((long long)nqb * part / p.units_per_pair);
    u.qb1 = (int)((long long)nqb * (part + 1) / p.units_per_pair);
    if (p.frame_rows[pd.t_frame] < 1) u.qb1 = u.qb0;  // nothing to compare against
    return u;
}

}  // namespace

constexpr int kScratchStride = 20;          // floats per lane (16 used; 80-byte stride keeps STS.128 conflict-free)
constexpr int kStageFloats = kTileFloats + kTile;   // tile + the 128 column thresholds that travel with it
constexpr int kStageBytes = kStageFloats * 4;

// Two smallest of a value replicated over a lane group by xor-shuffles: (lo, hi) <- merge with partner's (lo, hi).
__device__ __forceinline__ void merge_lo_hi(float& lo, float& hi, int xor_mask) {
    const float plo = __shfl_xor_sync(0xffffffffu, lo, xor_mask);
    const float phi = __shfl_xor_sync(0xffffffffu, hi, xor_mask);
    hi = fminf(fmaxf(lo, plo), fminf(hi, phi));
    lo = fminf(lo, plo);
}

// Lane-private sorted pair of row candidates, ordered by (value, index).  Within a lane the columns of a row
// arrive in ascending index order, so a strict '<' on the value keeps the lowest index among equal values.
struct RowTop2 {
    float v1, v2;
    uint32_t i1, i2;
};
__device__ __forceinline__ void row_insert(RowTop2& r, float v, uint32_t idx) {
    if (v < r.v2) {
        if (v < r.v1) {
            r.v2 = r.v1; r.i2 = r.i1;
            r.v1 = v;    r.i1 = idx;
        } else {
            r.v2 = v;    r.i2 = idx;
        }
    }
}
// Merge with the partner lane's pair (lexicographic on (value, index): lanes hold disjoint column sets).
__device__ __forceinline__ bool key_less(float va, uint32_t ia, float vb, uint32_t ib) { return va < vb || (va == vb && ia < ib); }
__device__ __forceinline__ void row_merge_xor(RowTop2& r, int xor_mask) {
    const float pv1 = __shfl_xor_sync(0xffffffffu, r.v1, xor_mask), pv2 = __shfl_xor_sync(0xffffffffu, r.v2, xor_mask);
    const uint32_t pi1 = __shfl_xor_sync(0xffffffffu, r.i1, xor_mask), pi2 = __shfl_xor_sync(0xffffffffu, r.i2, xor_mask);
    RowTop2 o;
    if (key_less(pv1, pi1, r.v1, r.i1)) {       // partner's best wins
        o.v1 = pv1; o.i1 = pi1;
        if (key_less(pv2, pi2, r.v1, r.i1)) { o.v2 = pv2; o.i2 = pi2; } else { o.v2 = r.v1; o.i2 = r.i1; }
    } else {
        o.v1 = r.v1; o.i1 = r.i1;
        if (key_less(pv1, pi1, r.v2, r.i2)) { o.v2 = pv1; o.i2 = pi1; } else { o.v2 = r.v2; o.i2 = r.i2; }
    }
    r = o;
}

template <int STAGES>
__global__ void __launch_bounds__(kSweepThreads, 1) sweep_l2_kernel(const SweepParams p) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    float* Qs = reinterpret_cast<float*>(smem_raw);                       // kQTiles tiles
    float* Ts = Qs + kQTiles * kTileFloats;                               // STAGES x (tile + 128 column thresholds)
    uint64_t* bars = reinterpret_cast<uint64_t*>(Ts + STAGES * kStageFloats);
    uint64_t* fullQ = bars;
    uint64_t* emptyQ = bars + 1;
    uint64_t* fullT = bars + 2;
    uint64_t* emptyT = bars + 2 + STAGES;
    float* scratch = reinterpret_cast<float*>(bars + 2 + 2 * STAGES);     // 256 lanes x kScratchStride
    float4* rowstate = reinterpret_cast<float4*>(scratch + kConsumerThreads * kScratchStride);  // [8 rows][256 lanes] (v1, v2, i1, i2)

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n_units = p.n_pairs * p.units_per_pair;

    if (threadIdx.x == 0) {
        mbar_init(fullQ, 1);
        mbar_init(emptyQ, kConsumerThreads / 32);
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(&fullT[s], 1);
            mbar_init(&emptyT[s], kConsumerThreads / 32);
        }
        fence_mbar_init();
    }
    __syncthreads();

    if (warp >= kConsumerThreads / 32) {
        // ============ producer warpgroup: one lane drives the TMA bulk copies, the rest idle ============
        reg_dealloc<40>();
        if (threadIdx.x == kConsumerThreads) {
            uint32_t g = 0, qseq = 0;
            for (int unit = blockIdx.x; unit < n_units; unit += gridDim.x) {
                const UnitInfo u = decode_unit(p, unit);
                const float* qbase = p.kmajor + (size_t)p.frame_tile_off[u.q_frame] * kTileFloats;
                const float* tbase = p.kmajor + (size_t)p.frame_tile_off[u.t_frame] * kTileFloats;
                const uint32_t* tauc = p.col_thr + (size_t)u.pair * p.stride;
                for (int qb = u.qb0; qb < u.qb1; ++qb) {
                    const int ntq = min(kQTiles, u.nqt - qb * kQTiles);
                    mbar_wait_backoff(emptyQ, (qseq & 1) ^ 1);
                    mbar_arrive_expect_tx(fullQ, (uint32_t)ntq * kTileBytes);
                    bulk_g2s(Qs, qbase + (size_t)qb * kQTiles * kTileFloats, (uint32_t)ntq * kTileBytes, fullQ);
                    ++qseq;
                    for (int tt = 0; tt < u.ntt; ++tt, ++g) {
                        const uint32_t st = g % STAGES, ph = (g / STAGES) & 1;
                        mbar_wait_backoff(&emptyT[st], ph ^ 1);
                        mbar_arrive_expect_tx(&fullT[st], kStageBytes);
                        float* dst = Ts + (size_t)st * kStageFloats;
                        bulk_g2s(dst, tbase + (size_t)tt * kTileFloats, kTileBytes, &fullT[st]);
                        // the running column thresholds of this tile ride along (a snapshot a few tiles old is fine:
                        // a stale threshold is only looser, never wrong)
                        bulk_g2s(dst + kTileFloats, tauc + (size_t)tt * kTile, kTile * 4, &fullT[st]);
                    }
                }
            }
        }
        return;
    }

    // ================================ consumer warps ================================
    reg_alloc<232>();
    const int qt = warp >> 2;                          // which of the 2 query tiles this warp works on
    const int ty = ((warp & 3) << 2) | (lane >> 3);    // 0..15 : row group inside the tile
    const int tx = lane & 7;                           // 0..7  : column group
    // rows of this thread inside the tile: r(i) = (i>>2)*64 + ty*4 + (i&3), i < 8
    // cols of this thread inside the tile: c(j) = (j>>2)*32 + tx*4 + (j&3), j < 16
    float* myscr = scratch + threadIdx.x * kScratchStride;
    float4* mystate = rowstate + threadIdx.x;   // row i of this lane lives at mystate[i * 256]: conflict-free 16-byte accesses
    uint32_t g = 0, qseq = 0;
    for (int unit = blockIdx.x; unit < n_units; unit += gridDim.x) {
        const UnitInfo u = decode_unit(p, unit);
        u64* rk1 = p.keys + (size_t)u.pair * 4 * p.stride;
        u64* rk2 = rk1 + p.stride;
        u64* ck1 = rk2 + p.stride;
        uint32_t* tauc = p.col_thr + (size_t)u.pair * p.stride;   // column thresholds of this pair (global, shared by all CTAs)

        for (int qb = u.qb0; qb < u.qb1; ++qb) {
            const int ntq = min(kQTiles, u.nqt - qb * kQTiles);
            const bool active = qt < ntq;
            mbar_wait(fullQ, qseq & 1);
            ++qseq;
            const float* Qt = Qs + qt * kTileFloats;
            float tr[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                tr[i] = __uint_as_float(kThrInit);     // shared (8 lanes of the row) running bound on the row's 2nd best
                mystate[i * kConsumerThreads] = make_float4(__int_as_float(0x7f800000), __int_as_float(0x7f800000),
                                                            __int_as_float(-1), __int_as_float(-1));
            }
            const int qrow0 = qb * (kQTiles * kTile) + qt * kTile;  // frame row of this warp's tile row 0
            const int row0 = qrow0 + ty * 4;

            for (int tt = 0; tt < u.ntt; ++tt, ++g) {
                const uint32_t st = g % STAGES, ph = (g / STAGES) & 1;
                mbar_wait(&fullT[st], ph);
                if (active) {
                    const float* Tt = Ts + (size_t)st * kStageFloats;
                    float2 acc[8][8];
                    {   // acc = hq_i + ht_j   (one packed op per pair)
                        float hq[8];
                        {
                            const float4 h0 = lds128(Qt + kDim * kTile + ty * 4), h1 = lds128(Qt + kDim * kTile + 64 + ty * 4);
                            hq[0] = h0.x; hq[1] = h0.y; hq[2] = h0.z; hq[3] = h0.w;
                            hq[4] = h1.x; hq[5] = h1.y; hq[6] = h1.z; hq[7] = h1.w;
                        }
                        float ht[16];
#pragma unroll
                        for (int m = 0; m < 4; ++m) {
                            const float4 h = lds128(Tt + kDim * kTile + m * 32 + tx * 4);
                            ht[m * 4 + 0] = h.x; ht[m * 4 + 1] = h.y; ht[m * 4 + 2] = h.z; ht[m * 4 + 3] = h.w;
                        }
                        const float2 one = make_float2(1.f, 1.f);
#pragma unroll
                        for (int i = 0; i < 8; ++i)
#pragma unroll
                            for (int jp = 0; jp < 8; ++jp)
                                acc[i][jp] = __ffma2_rn(make_float2(hq[i], hq[i]), one, make_float2(ht[2 * jp], ht[2 * jp + 1]));
                    }
                    const float* qp = Qt + ty * 4;
                    const float* tp = Tt + tx * 4;
#pragma unroll 8
                    for (int k = 0; k < kDim; ++k) {
                        const float4 a0 = lds128(qp + k * kTile), a1 = lds128(qp + k * kTile + 64);
                        const float4 b0 = lds128(tp + k * kTile), b1 = lds128(tp + k * kTile + 32);
                        const float4 b2 = lds128(tp + k * kTile + 64), b3 = lds128(tp + k * kTile + 96);
                        const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
                        const float2 b[8] = {make_float2(b0.x, b0.y), make_float2(b0.z, b0.w), make_float2(b1.x, b1.y),
                                             make_float2(b1.z, b1.w), make_float2(b2.x, b2.y), make_float2(b2.z, b2.w),
                                             make_float2(b3.x, b3.y), make_float2(b3.z, b3.w)};
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
                            const float na = -a[i];
#pragma unroll
                            for (int jp = 0; jp < 8; ++jp) {
                                unsigned long long& c = *reinterpret_cast<unsigned long long*>(&acc[i][jp]);
                                const unsigned long long bb = *reinterpret_cast<const unsigned long long*>(&b[jp]);
                                asm("{ .reg .b64 aa; mov.b64 aa, {%2, %2}; fma.rn.f32x2 %0, aa, %1, %0; }" : "+l"(c) : "l"(bb), "f"(na));
                            }
                        }
                    }

                    // ---------------- epilogue, fast path: minima (3-input FMNMX trees) vs thresholds ----------------
                    float tc[16], rm[8], cm[16];
#pragma unroll
                    for (int m = 0; m < 4; ++m) {
                        const float4 t = lds128(Tt + kTileFloats + m * 32 + tx * 4);
                        tc[m * 4 + 0] = t.x; tc[m * 4 + 1] = t.y; tc[m * 4 + 2] = t.z; tc[m * 4 + 3] = t.w;
                    }
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        float m = fminf(acc[i][0].x, acc[i][0].y);
#pragma unroll
                        for (int jp = 1; jp < 8; ++jp) m = fminf(fminf(m, acc[i][jp].x), acc[i][jp].y);
                        rm[i] = m;
                    }
#pragma unroll
                    for (int jp = 0; jp < 8; ++jp) {
                        float mx = fminf(acc[0][jp].x, acc[1][jp].x), my = fminf(acc[0][jp].y, acc[1][jp].y);
#pragma unroll
                        for (int i = 2; i < 8; i += 2) {
                            mx = fminf(fminf(mx, acc[i][jp].x), acc[i + 1][jp].x);
                            my = fminf(fminf(my, acc[i][jp].y), acc[i + 1][jp].y);
                        }
                        cm[2 * jp] = mx;
                        cm[2 * jp + 1] = my;
                    }
                    const int col0 = tt * kTile + tx * 4;
                    // The first tile of a query block has no row bound yet.  Seed one from the tile itself so that only
                    // O(2) elements per row go down the slow path: the second smallest of the 8 lane minima is >= the
                    // row's true second smallest, hence a valid (conservative) bound.
                    if (tt == 0) {
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
                            float lo = rm[i], hi = __uint_as_float(kThrInit);
                            merge_lo_hi(lo, hi, 1); merge_lo_hi(lo, hi, 2); merge_lo_hi(lo, hi, 4);
                            tr[i] = hi;
                        }
                    }
                    uint32_t mymask = 0;
#pragma unroll
                    for (int i = 0; i < 8; ++i) mymask |= (rm[i] <= tr[i]) ? (1u << i) : 0u;
#pragma unroll
                    for (int j = 0; j < 16; ++j) mymask |= (cm[j] <= tc[j]) ? (256u << j) : 0u;
                    const uint32_t wmask = __reduce_or_sync(0xffffffffu, mymask);

                    // ---------------- slow path: ~2 ln F hits per row, ~ln F per column over a whole sweep ----------------
                    // Visit only the bodies (8 rows, 16 columns of the register tile) some lane flagged.  The switch is the
                    // only per-body static code: it copies the flagged lane's 16 (row) or 8 (column) accumulators to its
                    // private shared-memory line; everything else is ONE generic routine working on that line, so the whole
                    // slow path is a few hundred instructions and stays resident in the instruction cache.
                    if (wmask) {
                        uint32_t todo = wmask;
#pragma unroll 1
                        while (todo) {
                            const int b = __ffs(todo) - 1;
                            todo &= todo - 1;
                            const bool flagged = (mymask >> b) & 1;
                            float thr = 0.f, vmin = 0.f;
                            switch (b) {
#define ROW_CASE(i)                                                                                                     \
    case i:                                                                                                             \
        thr = tr[i]; vmin = rm[i];                                                                                      \
        if (flagged) {                                                                                                  \
            _Pragma("unroll") for (int m = 0; m < 4; ++m)                                                               \
                *reinterpret_cast<float4*>(myscr + 4 * m) = make_float4(acc[i][2 * m].x, acc[i][2 * m].y, acc[i][2 * m + 1].x, acc[i][2 * m + 1].y); \
        }                                                                                                               \
        break;
                                ROW_CASE(0) ROW_CASE(1) ROW_CASE(2) ROW_CASE(3) ROW_CASE(4) ROW_CASE(5) ROW_CASE(6) ROW_CASE(7)
#undef ROW_CASE
#define COL_CASE(j)                                                                                                     \
    case 8 + j:                                                                                                         \
        thr = tc[j]; vmin = cm[j];                                                                                      \
        if (flagged) {                                                                                                  \
            *reinterpret_cast<float4*>(myscr) = (j & 1) ? make_float4(acc[0][j >> 1].y, acc[1][j >> 1].y, acc[2][j >> 1].y, acc[3][j >> 1].y)      \
                                                          : make_float4(acc[0][j >> 1].x, acc[1][j >> 1].x, acc[2][j >> 1].x, acc[3][j >> 1].x);     \
            *reinterpret_cast<float4*>(myscr + 4) = (j & 1) ? make_float4(acc[4][j >> 1].y, acc[5][j >> 1].y, acc[6][j >> 1].y, acc[7][j >> 1].y)  \
                                                              : make_float4(acc[4][j >> 1].x, acc[5][j >> 1].x, acc[6][j >> 1].x, acc[7][j >> 1].x); \
        }                                                                                                               \
        break;
                                COL_CASE(0) COL_CASE(1) COL_CASE(2) COL_CASE(3) COL_CASE(4) COL_CASE(5) COL_CASE(6) COL_CASE(7)
                                COL_CASE(8) COL_CASE(9) COL_CASE(10) COL_CASE(11) COL_CASE(12) COL_CASE(13) COL_CASE(14) COL_CASE(15)
#undef COL_CASE
                                default: break;
                            }
                            if (!flagged) continue;
                            if (b < 8) {
                                // ---- generic row routine: lane-private top-2 of row b over this lane's columns ----
                                const float4 v0 = *reinterpret_cast<const float4*>(myscr), v1 = *reinterpret_cast<const float4*>(myscr + 4);
                                const float4 v2 = *reinterpret_cast<const float4*>(myscr + 8), v3 = *reinterpret_cast<const float4*>(myscr + 12);
                                const float v[16] = {v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w, v2.x, v2.y, v2.z, v2.w, v3.x, v3.y, v3.z, v3.w};
                                uint32_t hm = 0;
#pragma unroll
                                for (int k = 0; k < 16; ++k) hm |= (v[k] <= thr) ? (1u << k) : 0u;
                                float4* sp = mystate + b * kConsumerThreads;
                                const float4 st4 = *sp;
                                RowTop2 t;
                                t.v1 = st4.x; t.v2 = st4.y; t.i1 = __float_as_uint(st4.z); t.i2 = __float_as_uint(st4.w);
                                if (__builtin_expect((hm & (hm - 1)) == 0, 1)) {
                                    const int k = __ffs(hm) - 1;
                                    row_insert(t, vmin, (uint32_t)(col0 + (k >> 2) * 32 + (k & 3)));
                                } else {
                                    while (hm) {
                                        const int k = __ffs(hm) - 1;
                                        hm &= hm - 1;
                                        row_insert(t, myscr[k], (uint32_t)(col0 + (k >> 2) * 32 + (k & 3)));
                                    }
                                }
                                *sp = make_float4(t.v1, t.v2, __uint_as_float(t.i1), __uint_as_float(t.i2));
                            } else {
                                // ---- generic column routine: fire-and-forget 64-bit min on the packed key (value bits << 32 |
                                // query row) and 32-bit min on the running threshold: no return value, nothing waits on L2 ----
                                const float4 v0 = *reinterpret_cast<const float4*>(myscr), v1 = *reinterpret_cast<const float4*>(myscr + 4);
                                const float v[8] = {v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w};
                                uint32_t hm = 0;
#pragma unroll
                                for (int k = 0; k < 8; ++k) hm |= (v[k] <= thr) ? (1u << k) : 0u;
                                const int jj = b - 8;
                                const uint32_t gcol = (uint32_t)(col0 + (jj >> 2) * 32 + (jj & 3));
                                if (__builtin_expect((hm & (hm - 1)) == 0, 1)) {
                                    const int k = __ffs(hm) - 1;
                                    atomicMin(ck1 + gcol, make_key(__float_as_uint(fmaxf(vmin, 0.f)), (uint32_t)(row0 + (k >> 2) * 64 + (k & 3))));
                                } else {
                                    while (hm) {
                                        const int k = __ffs(hm) - 1;
                                        hm &= hm - 1;
                                        atomicMin(ck1 + gcol, make_key(__float_as_uint(fmaxf(myscr[k], 0.f)), (uint32_t)(row0 + (k >> 2) * 64 + (k & 3))));
                                    }
                                }
                                atomicMin(tauc + gcol, __float_as_uint(fmaxf(vmin, 0.f)));
                            }
                        }
                        if (wmask & 0xffu) {
                            // refresh the shared bound of every row: exact second best over its 8 lanes' candidate pairs
                            // (8 independent shuffle chains, so their latencies overlap)
                            __syncwarp();
                            float lo[8], hi[8];
#pragma unroll
                            for (int i = 0; i < 8; ++i) {
                                const float2 s2 = *reinterpret_cast<const float2*>(&mystate[i * kConsumerThreads]);
                                lo[i] = s2.x; hi[i] = s2.y;
                            }
#pragma unroll
                            for (int x = 1; x <= 4; x <<= 1)
#pragma unroll
                                for (int i = 0; i < 8; ++i) merge_lo_hi(lo[i], hi[i], x);
#pragma unroll
                            for (int i = 0; i < 8; ++i) tr[i] = fminf(tr[i], hi[i]);
                        }
                    }
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(&emptyT[st]);
            }
            // ---- end of the sweep for this query block: merge the 8 lanes of every row and publish its two candidates ----
            if (active) {
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const float4 st4 = mystate[i * kConsumerThreads];
                    RowTop2 t;
                    t.v1 = st4.x; t.v2 = st4.y; t.i1 = __float_as_uint(st4.z); t.i2 = __float_as_uint(st4.w);
                    row_merge_xor(t, 1); row_merge_xor(t, 2); row_merge_xor(t, 4);
                    if (tx == 0) {
                        const int grow = row0 + (i >> 2) * 64 + (i & 3);
                        rk1[grow] = t.i1 == 0xffffffffu ? kKeyInit : make_key(__float_as_uint(fmaxf(t.v1, 0.f)), t.i1);
                        rk2[grow] = t.i2 == 0xffffffffu ? kKeyInit : make_key(__float_as_uint(fmaxf(t.v2, 0.f)), t.i2);
                    }
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(emptyQ);
        }
    }
}

size_t sweep_l2_smem_bytes(int stages) {
    return (size_t)kQTiles * kTileBytes + (size_t)stages * kStageBytes + (2 + 2 * stages) * 8 +
           (size_t)kConsumerThreads * kScratchStride * 4 + (size_t)8 * kConsumerThreads * sizeof(float4);
}

int sweep_l2_max_rows() { return (1 << 20) / kTile * kTile; }

cudaError_t launch_sweep_l2(const SweepParams& p, int sm_count, cudaStream_t s) {
    const int n_units = p.n_pairs * p.units_per_pair;
    if (n_units <= 0) return cudaSuccess;
    const int grid = n_units < sm_count ? n_units : sm_count;
    constexpr int kStages = 3;
    const size_t smem = sweep_l2_smem_bytes(kStages);
    cudaError_t e = cudaFuncSetAttribute(sweep_l2_kernel<kStages>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    sweep_l2_kernel<kStages><<<grid, kSweepThreads, smem, s>>>(p);
    return cudaGetLastError();
}

}  // namespace esfm
