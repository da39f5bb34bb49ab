// finalize.cu -- per image pair: exact re-evaluation of the surviving candidates, Lowe ratio test,
// mutual cross-check and stable compaction into the dense match arena.
//
// Replaces the reference's ratio loop  cpp_code/src/feature_matching.cpp:84-92 / :129-137
//   if (nn[i][0].distance < ratio_thre * nn[i][1].distance) matches.push_back(nn[i][0]);
// (float distances promoted to double, `double ratio_thre` from feature_matching.h:17-21) and the
// crossCheck=True filter of python_code/feature_match.py:26-27.  Output order = ascending queryIdx,
// imgIdx = 0, exactly what push_back inside `for i` over the queries produces.
//
// L2: the sweep ranks with the expansion 1/2|q|^2 + 1/2|t|^2 - q.t, whose fp32 cancellation error is too
// large to REPORT (SURVEY.md F10).  Here the two row candidates -- and, for the cross-check, the two
// column candidates of the chosen train row -- are recomputed in direct form sum (a-b)^2 with the
// summation order fixed in oracle/bf_oracle.c and re-ordered by (distance, index).
// Hamming: the sweep's integer distances are already exact.
#include "esfm_internal.cuh"

namespace esfm {

namespace {

constexpr int kFinThreads = 256;
constexpr int kFinBuckets = 1024;      // two-phase cross-check: histogram buckets of the sweep's ranking values
// ORB: value = 2 * hamming -> bucket = hamming (exact); SURF: value = 1/2 d^2 in [0, 2] for unit-norm rows -> 512 buckets per unit,
// everything beyond in the last one (conservative: a coarser bucket only sends more train rows to the verification sweep)
template <int KIND> __device__ __forceinline__ int fin_bucket(float v) {
    if (KIND == ESFM_KIND_B256) return min(kFinBuckets - 1, max(0, (int)(0.5f * v)));
    return min(kFinBuckets - 1, max(0, (int)(v * 512.f)));
}

struct RowResult {
    int t1;
    float d1;
    float d2;       // SURF slice keys: the second of the columns finalize evaluated (+inf: none), a bound for histogram B
    bool keep;
};

__device__ __forceinline__ void order2(float& da, int& ia, float& db, int& ib) {
    // ascending by (distance, index)
    if (db < da || (db == da && ib < ia)) {
        const float td = da; da = db; db = td;
        const int ti = ia; ia = ib; ib = ti;
    }
}

// Hamming distance out of the high word of a sweep key (KeyFormat)
__device__ __forceinline__ float b256_key_distance(const FinalizeParams& p, u64 k) {
    const uint32_t hi = (uint32_t)(k >> 32);
    if (p.key_format == KeyFormat::TcZ) return (float)(((int)__uint_as_float(hi) - kTcZ0i) >> kTcZShift);
    if (p.key_format == KeyFormat::TcPm1) return 0.5f * __uint_as_float(hi);
    return (float)hi;      // Direct (slice keys are read by eval_rows_win)
}

template <int KIND>
__device__ __forceinline__ RowResult eval_row(const FinalizeParams& p, const u64* rk1, const u64* rk2, const u64* ck1,
                                              const float* qrows, const float* trows, int q, int32_t* knn_idx, float* knn_dist) {
    RowResult r;
    r.keep = false;
    r.t1 = -1;
    r.d1 = 0.f;
    r.d2 = __int_as_float(0x7f800000);
    const u64 k1 = rk1[q], k2 = rk2[q];
    int i1 = -1, i2 = -1;
    float d1 = __int_as_float(0x7f800000), d2 = d1;
    if (k1 != kKeyInit) {
        i1 = (int)(uint32_t)k1;
        if (KIND == ESFM_KIND_F32X64) d1 = l2_direct(qrows + (size_t)q * kDim, trows + (size_t)i1 * kDim);
        else d1 = b256_key_distance(p, k1);
    }
    if (k2 != kKeyInit) {
        i2 = (int)(uint32_t)k2;
        if (KIND == ESFM_KIND_F32X64) {
            d2 = l2_direct(qrows + (size_t)q * kDim, trows + (size_t)i2 * kDim);
            order2(d1, i1, d2, i2);
        } else {
            d2 = b256_key_distance(p, k2);
        }
    }
    if (knn_idx) {
        knn_idx[2 * q] = i1; knn_idx[2 * q + 1] = i2;
        knn_dist[2 * q] = d1; knn_dist[2 * q + 1] = d2;
    }
    if (p.ratio == __longlong_as_double(0x7ff0000000000000LL)) {
        // ratio = +inf: no ratio test (plain mutual-NN matching, python_code/feature_match.py:26-27)
        if (i1 < 0) return r;
    } else {
        if (i2 < 0) return r;  // fewer than two neighbours: the reference has no defined behaviour, we emit nothing (F7)
        if (!((double)d1 < p.ratio * (double)d2)) return r;
    }
    if (p.cross_check) {
        // nearest query row of train row i1 (lowest index on ties) must be q
        const u64 c1 = ck1[i1];
        if (c1 == kKeyInit) return r;
        const int best = (int)(uint32_t)c1;
        if (best != q) {
            if (KIND != ESFM_KIND_F32X64) return r;
            // The sweep ranked the column in expansion form; q may still be the true nearest row if the two are
            // within its rounding noise.  Decide in direct form, (distance, index) order.
            const float db = l2_direct(qrows + (size_t)best * kDim, trows + (size_t)i1 * kDim);
            if (!(d1 < db || (d1 == db && q < best))) return r;
        }
    }
    r.keep = true;
    r.t1 = i1;
    r.d1 = d1;
    return r;
}

// ---- slice keys (sweep_win.cu): a row key's low word names a slice of train columns instead of one column ----
//     id = (first column / 8) << 2 | width code         0: 8 columns, 1: 32, 2: 64, 3: 128      (| kWinExactMark: see SweepParams::fallback)
// The column itself is found HERE, by evaluating the slice exactly -- and only for rows that can still pass the ratio test.
__device__ __forceinline__ void win_range(u64 key, int ft, int& c0, int& c1) {
    const uint32_t id = (uint32_t)key & ~kWinExactMark;
    c0 = (int)(id >> 2) * 8;
    const uint32_t w = id & 3u;
    c1 = min(c0 + (w == 0u ? 8 : (w == 1u ? 32 : (w == 2u ? 64 : 128))), ft);
}
__device__ __forceinline__ int b256_hamming(const uint4& a0, const uint4& a1, const uint4* __restrict__ t) {
    const uint4 b0 = __ldg(t), b1 = __ldg(t + 1);
    return __popc(a0.x ^ b0.x) + __popc(a0.y ^ b0.y) + __popc(a0.z ^ b0.z) + __popc(a0.w ^ b0.w) +
           __popc(a1.x ^ b1.x) + __popc(a1.y ^ b1.y) + __popc(a1.z ^ b1.z) + __popc(a1.w ^ b1.w);
}
// lowest column of [c0, c1) at Hamming distance `want` from the query row, skipping column `skip`
__device__ __forceinline__ int b256_find(const uint4& a0, const uint4& a1, const uint4* __restrict__ tbits, int c0, int c1, int want, int skip) {
    for (int c = c0; c < c1; ++c)
        if (c != skip && b256_hamming(a0, a1, tbits + (size_t)c * 2) == want) return c;
    return -1;
}
// exact top-2 by (distance, index) of the columns [c0, c1) merged into (d1, i1, d2, i2)
__device__ __forceinline__ void l2_scan(const float* __restrict__ qrow, const float* __restrict__ trows, int c0, int c1, float& d1, int& i1, float& d2, int& i2) {
    for (int c = c0; c < c1; ++c) {
        const float d = l2_direct(qrow, trows + (size_t)c * kDim);
        if (d < d1 || (d == d1 && c < i1)) {
            d2 = d1; i2 = i1;
            d1 = d; i1 = c;
        } else if (d < d2 || (d == d2 && c < i2)) {
            d2 = d; i2 = c;
        }
    }
}

// lexicographic (distance, index) merge of another sorted pair (e1, j1) <= (e2, j2) into (d1, i1) <= (d2, i2)
__device__ __forceinline__ void top2_merge(float& d1, int& i1, float& d2, int& i2, float e1, int j1, float e2, int j2) {
    const bool other_first = e1 < d1 || (e1 == d1 && j1 < i1);
    const float a1 = other_first ? e1 : d1, b1 = other_first ? d1 : e1;           // a = the winner's side, b = the loser's best
    const int ai = other_first ? j1 : i1, bi = other_first ? i1 : j1;
    const float a2 = other_first ? e2 : d2;                                          // the winner's own second
    const int a2i = other_first ? j2 : i2;
    const bool loser_second = b1 < a2 || (b1 == a2 && bi < a2i);
    d1 = a1; i1 = ai;
    d2 = loser_second ? b1 : a2;
    i2 = loser_second ? bi : a2i;
}

// The 32 rows of one warp iteration (row q per lane; `valid` lanes only), slice keys.  WARP-COOPERATIVE: the rows that need their slice
// evaluated are served four at a time by groups of eight lanes -- one candidate column per lane and step, all loads of a step in flight
// together -- instead of every lane walking its own slice serially (a quarter of the lanes busy, eight dependent gathers each: that walk
// was 90 % of the kernel's time).  Each distance is still computed by ONE lane with l2_direct (the oracle's summation order).
// `e`: SURF, the row's values come from the fast sweep and are within e of the exact ones (0: exact mode).
template <int KIND>
__device__ __forceinline__ RowResult eval_rows_win(const FinalizeParams& p, u64 k1, u64 k2, float e, const float* qrows, const float* trows,
                                                   const uint4* qbits, const uint4* tbits, int q, int ft, bool valid) {
    const unsigned full = 0xffffffffu;
    const int lane = threadIdx.x & 31, grp = lane >> 3, sub = lane & 7;
    const bool has1 = valid && k1 != kKeyInit, has2 = valid && k2 != kKeyInit;
    const bool no_ratio = p.ratio == __longlong_as_double(0x7ff0000000000000LL);
    const float inf = __int_as_float(0x7f800000);
    int i1 = -1, i2 = -1;
    float d1 = inf, d2 = inf;
    bool pass = false, scan_a = false, scan_b = false, exact_ratio = false;
    int a0 = 0, a1 = 0, b0 = 0, b1 = 0;
    if (has1) win_range(k1, ft, a0, a1);
    if (has2) win_range(k2, ft, b0, b1);
    if (KIND == ESFM_KIND_B256) {
        // the sweep's integer distances are exact: only the column has to be found, and only for rows that pass
        if (has1) d1 = 0.5f * __uint_as_float((uint32_t)(k1 >> 32));
        if (has2) d2 = 0.5f * __uint_as_float((uint32_t)(k2 >> 32));
        pass = has1 && (no_ratio || (has2 && (double)d1 < p.ratio * (double)d2));
        scan_a = pass;
    } else if (has1) {
        // CHAIN keys: k1 = the best chain of 8 columns (its maximum is the row's best value s1), k2 = the second chain, whose value s2 is
        // the best of every column outside the best chain.  The true second lies in one of the two chains, and s2 >= it: a certain fail
        // on (s1, s2) is certain, a certain pass only says that the columns outside the best chain cannot fail the row -- the best
        // chain's own second, evaluated below, must pass the exact test too.  No second chain (the train frame fits one chain, or every
        // other chain is pad): s2 = +inf, and the best chain's own second decides.  The sweep's values are within ~4e-7 absolute of the
        // expansion form (or within e): decide far-from-the-boundary rows on them, evaluate the rest -- and every reported distance --
        // in direct form.  (A fast-mode row never lands in between: win_classify has sent those to the fallback sweep.)
        const float s1 = __uint_as_float((uint32_t)(k1 >> 32)), s2 = has2 ? __uint_as_float((uint32_t)(k2 >> 32)) : inf;
        if (no_ratio) { pass = true; scan_a = true; }
        else if (p.ratio > 0.0) {
            const int cls = win_ratio_class(s1, s2, e, (float)(p.ratio * p.ratio));
            if (cls != 0) {
                scan_a = true;
                pass = cls == 1;
                if (cls == 2) { scan_b = true; exact_ratio = true; }     // (s2 = +inf is never class 2: has2 holds here)
            }
        }
        if (scan_b && a0 >= b0 && a1 <= b1) scan_a = false;       // slice a lies inside slice b: one evaluation
    }
    // ---- the cooperative part: four flagged rows per round, eight lanes each ----
    unsigned todo = __ballot_sync(full, scan_a || scan_b);
    while (todo) {
        // owner lanes of this round's four rows (-1: none)
        int owner[4];
        unsigned rest = todo;
#pragma unroll
        for (int g = 0; g < 4; ++g) {
            owner[g] = rest ? __ffs(rest) - 1 : -1;
            rest &= rest - 1;
        }
        todo = rest;
        const int mine_owner = grp == 0 ? owner[0] : (grp == 1 ? owner[1] : (grp == 2 ? owner[2] : owner[3]));
        const int src = mine_owner < 0 ? 0 : mine_owner;
        const bool active = mine_owner >= 0;
        const int rq = __shfl_sync(full, q, src);
        const int ra0 = __shfl_sync(full, scan_a ? a0 : 0, src), ra1 = __shfl_sync(full, scan_a ? a1 : 0, src);
        const int rb0 = __shfl_sync(full, scan_b ? b0 : 0, src), rb1 = __shfl_sync(full, scan_b ? b1 : 0, src);
        if (KIND == ESFM_KIND_B256) {
            const int want = (int)__shfl_sync(full, d1, src);
            uint4 q0 = make_uint4(0, 0, 0, 0), q1 = q0;
            if (active) { q0 = __ldg(qbits + (size_t)rq * 2); q1 = __ldg(qbits + (size_t)rq * 2 + 1); }
            int found = -1;
            const int steps = __reduce_max_sync(full, active ? (ra1 - ra0 + 7) >> 3 : 0);
            for (int k = 0; k < steps; ++k) {
                const int c = ra0 + 8 * k + sub;
                const bool hit = active && c < ra1 && b256_hamming(q0, q1, tbits + (size_t)c * 2) == want;
                const unsigned m = (__ballot_sync(full, hit) >> (8 * grp)) & 0xffu;
                if (found < 0 && m) found = ra0 + 8 * k + __ffs(m) - 1;
            }
#pragma unroll
            for (int g = 0; g < 4; ++g) {
                const int v = __shfl_sync(full, found, 8 * g);
                if (lane == owner[g]) i1 = v;
            }
        } else {
            float e1 = inf, e2 = inf;
            int j1 = -1, j2 = -1;
            const float* qrow = qrows + (size_t)rq * kDim;
#pragma unroll 1
            for (int part = 0; part < 2; ++part) {
                const int c0 = part ? rb0 : ra0, c1 = part ? rb1 : ra1;
                const int steps = __reduce_max_sync(full, active ? (c1 - c0 + 7) >> 3 : 0);
                for (int k = 0; k < steps; ++k) {
                    const int c = c0 + 8 * k + sub;
                    if (active && c < c1) {
                        const float d = l2_direct(qrow, trows + (size_t)c * kDim);
                        if (d < e1 || (d == e1 && c < j1)) { e2 = e1; j2 = j1; e1 = d; j1 = c; }
                        else if (d < e2 || (d == e2 && c < j2)) { e2 = d; j2 = c; }
                    }
                }
            }
#pragma unroll
            for (int m = 1; m <= 4; m <<= 1) {
                const float o1 = __shfl_xor_sync(full, e1, m), o2 = __shfl_xor_sync(full, e2, m);
                const int p1 = __shfl_xor_sync(full, j1, m), p2 = __shfl_xor_sync(full, j2, m);
                if (p1 >= 0) {
                    if (j1 < 0) { e1 = o1; j1 = p1; e2 = o2; j2 = p2; }
                    else top2_merge(e1, j1, e2, j2, o1, p1, p2 >= 0 ? o2 : inf, p2 >= 0 ? p2 : 0x7fffffff);
                }
            }
            if (j2 == 0x7fffffff) j2 = -1;
#pragma unroll
            for (int g = 0; g < 4; ++g) {
                const float v1 = __shfl_sync(full, e1, 8 * g), v2 = __shfl_sync(full, e2, 8 * g);
                const int w1 = __shfl_sync(full, j1, 8 * g), w2 = __shfl_sync(full, j2, 8 * g);
                if (lane == owner[g]) { d1 = v1; i1 = w1; d2 = v2; i2 = w2; }
            }
        }
    }
    if (KIND == ESFM_KIND_B256) {
        if (i1 < 0) pass = false;               // (cannot happen for a passing row: the sweep saw this distance in this slice)
    } else {
        // class 2: the exact top 2 of both chains; class 1: the best chain's own second (none: the second chain, which cannot fail)
        if (exact_ratio) pass = i2 >= 0 && (double)d1 < p.ratio * (double)d2;
        else if (pass && !no_ratio) pass = i2 >= 0 ? (double)d1 < p.ratio * (double)d2 : has2;
        if (i1 < 0) pass = false;
    }
    RowResult r;
    r.keep = pass;
    r.t1 = i1;
    r.d1 = d1;
    r.d2 = i2 >= 0 ? d2 : inf;
    return r;
}

// Two-phase cross-check, phase 2: is query row q (at exact distance d1) the nearest query row of train row t1, lowest index on ties?
// `vk` = what the verification sweep found for t1: (value bits, slice of QUERY rows holding the first row at the column minimum).
template <int KIND>
__device__ __forceinline__ bool verify_col(u64 vk, int q, int t1, float d1, const float* qrows, const float* trows, const uint4* qbits,
                                           const uint4* tbits, int fq) {
    if (vk == kKeyInit) return false;       // (cannot happen: the sweep saw at least row q)
    int c0, c1;
    win_range(vk, fq, c0, c1);
    if (KIND == ESFM_KIND_B256) {
        const float cv = 0.5f * __uint_as_float((uint32_t)(vk >> 32));
        if (cv < d1) return false;          // another query row is nearer
        if (cv > d1 || q < c0) return true; // (cannot happen: q itself is at d1)
        if (q >= c1) return false;          // the first row at this distance is in an earlier slice
        const uint4 t0 = __ldg(tbits + (size_t)t1 * 2), t1b = __ldg(tbits + (size_t)t1 * 2 + 1);
        for (int r = c0; r < q; ++r)
            if (b256_hamming(t0, t1b, qbits + (size_t)r * 2) == (int)d1) return false;
        return true;
    } else {
        // the sweep ranked the column in expansion form: decide between its winner's slice and q in direct form, (distance, index) order
        const float* trow = trows + (size_t)t1 * kDim;
        for (int r = c0; r < c1; ++r) {
            if (r == q) continue;
            const float d = l2_direct(qrows + (size_t)r * kDim, trow);
            if (d < d1 || (d == d1 && r < q)) return false;
        }
        return true;
    }
}

template <int KIND>
__global__ void __launch_bounds__(kFinThreads) finalize_kernel(const FinalizeParams p) {
    const int pair = blockIdx.x;
    const PairDesc pd = p.pairs[pair];
    const int fq = p.frame_rows[pd.q_frame], ft = p.frame_rows[pd.t_frame];
    u64* rk1 = p.keys + (size_t)pair * 4 * p.stride;
    u64* rk2 = rk1 + p.stride;
    const u64* ck1 = rk2 + p.stride;
    const u64* ck2 = ck1 + p.stride;
    const float* qrows = nullptr;
    const float* trows = nullptr;
    const uint4* qbits = nullptr;
    const uint4* tbits = nullptr;
    if (KIND == ESFM_KIND_F32X64) {
        qrows = p.rows_f32 + (size_t)p.frame_row_off[pd.q_frame] * kDim;
        trows = p.rows_f32 + (size_t)p.frame_row_off[pd.t_frame] * kDim;
    } else {
        qbits = p.rows_b256 + (size_t)p.frame_row_off[pd.q_frame] * 2;
        tbits = p.rows_b256 + (size_t)p.frame_row_off[pd.t_frame] * 2;
    }
    __shared__ unsigned int s_warp[kFinThreads / 32];
    __shared__ unsigned long long s_base;
    __shared__ unsigned int s_total;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;

    const bool no_ratio = p.ratio == __longlong_as_double(0x7ff0000000000000LL);
    __shared__ unsigned int s_targets;
    __shared__ unsigned int s_hist[2][kFinBuckets];
    if (fq == 0 || ft < (no_ratio ? 1 : 2)) {  // F7: no second neighbour exists
        if (p.phase == 1 && threadIdx.x == 0) p.gather_cnt[pair] = 0;
        if (p.knn_idx) {
            for (int q = threadIdx.x; q < fq; q += kFinThreads) {
                RowResult r = eval_row<KIND>(p, rk1, rk2, ck1, qrows, trows, q, p.knn_idx, p.knn_dist);     // (knn output: never slice keys)
                (void)r;
            }
        }
        if (threadIdx.x == 0) {
            p.pair_cnt[pair] = 0;
            p.pair_off[pair] = 0;
        }
        return;
    }

    // pass 1: evaluate every query row; stash the verdict in the row's first key slot
    unsigned int mine = 0;
    if (p.phase == 2) {
        // Two-phase cross-check, phase 2: the survivors of phase 1 against what the verification sweep found for their train rows
        // (ck1[t] = 2^40 | slot of train row t in the gather list, 4th key array [slot] = the sweep's answer)
        for (int q = threadIdx.x; q < fq; q += kFinThreads) {
            const u64 v = rk1[q];
            if (v == kKeyInit) continue;
            const int t1 = (int)(uint32_t)v;
            const float d1 = __uint_as_float((uint32_t)(v >> 32));
            if (rk2[q] == 1) { mine += 1u; continue; }           // decided in phase 1
            const u64 vk = ck2[(uint32_t)ck1[t1]];
            if (verify_col<KIND>(vk, q, t1, d1, qrows, trows, qbits, tbits, fq)) mine += 1u;
            else rk1[q] = kKeyInit;
        }
    } else {
    if (p.phase == 1) {
        for (int i = threadIdx.x; i < 2 * kFinBuckets; i += kFinThreads) (&s_hist[0][0])[i] = 0u;
        if (threadIdx.x == 0) s_targets = 0;
        __syncthreads();
    }
    if (p.key_format == KeyFormat::Slice) {
        const bool fast = KIND == ESFM_KIND_F32X64 && p.row_eps;
        const float* row_eps = fast ? p.row_eps + p.frame_row_off[pd.q_frame] : nullptr;
        const float nq = fast ? p.frame_norm[pd.q_frame] : 0.f, nt = fast ? p.frame_norm[pd.t_frame] : 0.f;
        // slice keys: every warp takes 32 consecutive rows per iteration and evaluates their slices cooperatively
        for (int q0 = warp * 32; q0 < fq; q0 += kFinThreads) {
            const int q = q0 + lane;
            const bool valid = q < fq;
            const u64 k1 = valid ? rk1[q] : kKeyInit, k2 = valid ? rk2[q] : kKeyInit;
            const float e = (fast && !((uint32_t)k1 & kWinExactMark)) ? win_fast_eps(row_eps[q], nq, nt) : 0.f;
            const RowResult r = eval_rows_win<KIND>(p, k1, k2, e, qrows, trows, qbits, tbits, q, ft, valid);
            if (!valid) continue;
            rk1[q] = r.keep ? make_key(__float_as_uint(r.d1), (uint32_t)r.t1) : kKeyInit;
            mine += r.keep ? 1u : 0u;
            if (p.phase == 1) {
                // Who could beat a survivor (q, t) at its own train row t?  A row whose NEAREST train row is t (another survivor: settled by
                // the claims below; a row that failed the ratio test: counted in histogram A by its best value), or a row for which t is at
                // best second (then its second-best value is <= its distance to t: histogram B takes a lower bound on every row's second
                // value).  A survivor whose distance lies below every such value needs no verification sweep.  Fast-mode values enter as
                // lower bounds, value - e: the k-th smallest of a row's values moves by at most e, whichever column the sweep named.
                // SURF chain keys: k2 is the best value OUTSIDE the best chain, so k2 - e bounds the true second only from above when the
                // second lies inside the best chain.  A survivor had its best chain evaluated exactly: its B entry is min(that chain's own
                // second, k2 - e).  A row that did not survive enters histogram A at k1 - e, below its second value: the prefix test
                // below only asks whether any entry lies at or below a value, so its B entry, never lower than its A entry, is dropped.
                if (KIND == ESFM_KIND_B256) {
                    if (k2 != kKeyInit) atomicAdd(&s_hist[1][fin_bucket<KIND>(__uint_as_float((uint32_t)(k2 >> 32)) - e)], 1u);
                } else if (r.keep) {
                    float lo2 = 0.5f * r.d2 * r.d2;     // (+inf: none)
                    if (k2 != kKeyInit) lo2 = fminf(lo2, __uint_as_float((uint32_t)(k2 >> 32)) - e);
                    if (lo2 != __int_as_float(0x7f800000)) atomicAdd(&s_hist[1][fin_bucket<KIND>(lo2)], 1u);
                }
                if (!r.keep && k1 != kKeyInit) atomicAdd(&s_hist[0][fin_bucket<KIND>(__uint_as_float((uint32_t)(k1 >> 32)) - e)], 1u);
                // every train row some survivor points at is claimed by the nearest such query row (lowest index on ties)
                if (r.keep) atomicMin(const_cast<u64*>(ck1) + r.t1, make_key(__float_as_uint(r.d1), (uint32_t)q));
            }
        }
    } else {
    for (int q = threadIdx.x; q < fq; q += kFinThreads) {
        const RowResult r = eval_row<KIND>(p, rk1, rk2, ck1, qrows, trows, q, p.knn_idx, p.knn_dist);
        rk1[q] = r.keep ? make_key(__float_as_uint(r.d1), (uint32_t)r.t1) : kKeyInit;
        mine += r.keep ? 1u : 0u;
    }
    }
    }
    if (p.phase == 1) {
        __syncthreads();
        // inclusive prefix sums of (A + B) over the buckets: s_hist[0][b] = rows that may be at least as near as bucket b
        if (warp == 0) {
            constexpr int kPer = kFinBuckets / 32;
            unsigned int loc = 0;
            for (int i = 0; i < kPer; ++i) loc += s_hist[0][lane * kPer + i] + s_hist[1][lane * kPer + i];
            unsigned int incl = loc;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const unsigned int o = __shfl_up_sync(0xffffffffu, incl, d);
                if (lane >= d) incl += o;
            }
            unsigned int run = incl - loc;
            for (int i = 0; i < kPer; ++i) {
                run += s_hist[0][lane * kPer + i] + s_hist[1][lane * kPer + i];
                s_hist[0][lane * kPer + i] = run;
            }
        }
        __syncthreads();
        // survivors: beaten by another survivor -> dropped; below every possible rival -> decided (state 1); else its train row goes on
        // the pair's list for the verification sweep (state 2; any order: the slot is looked up through ck1)
        int* gl = p.gather + (size_t)pair * p.stride;
        // SURF: the histograms hold the sweep's 1/2 d^2, whose error grows with the magnitudes the expansion form cancels,
        // m = 1/2 (nq^2 + nt^2) + nq nt (nq, nt: the frames' largest row norms, as in win_fast_eps) -- at norm 64 one ulp of a half norm
        // alone is 2.4e-4.  Compare with a margin of 2^-14 m (twice the rounding term win_fast_eps allows the 9-slot sweep; the exact
        // sweep has 13 slots), at least 1e-5.  Fast-mode rows entered the histograms at value - e already; the margin covers the rows
        // swept in exact mode (e = 0).  A larger margin only sends more train rows to the verification sweep.
        float margin = 1e-5f;
        if (KIND == ESFM_KIND_F32X64 && p.frame_norm) {
            const float nq = p.frame_norm[pd.q_frame], nt = p.frame_norm[pd.t_frame];
            margin = fmaxf(margin, 0x1p-14f * (0.5f * (nq * nq + nt * nt) + nq * nt));
        }
        for (int q = threadIdx.x; q < fq; q += kFinThreads) {
            const u64 v = rk1[q];
            if (v == kKeyInit) continue;
            const int t1 = (int)(uint32_t)v;
            const float d1 = __uint_as_float((uint32_t)(v >> 32));
            if (ck1[t1] != make_key((uint32_t)(v >> 32), (uint32_t)q)) { rk1[q] = kKeyInit; continue; }
            const float mine_v = KIND == ESFM_KIND_B256 ? 2.f * d1 : 0.5f * d1 * d1 + margin;
            if (s_hist[0][fin_bucket<KIND>(mine_v)] == 0u) { rk2[q] = 1; continue; }
            const unsigned int slot = atomicAdd(&s_targets, 1u);
            gl[slot] = t1;
            const_cast<u64*>(ck1)[t1] = (1ull << 40) | slot;
            rk2[q] = 2;
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            p.gather_cnt[pair] = (int)s_targets;
            if (s_targets) atomicAdd(p.verified_rows, (unsigned long long)s_targets);
        }
        return;
    }
    // block total -> one arena allocation per pair
    unsigned int wsum = __reduce_add_sync(0xffffffffu, mine);
    if (lane == 0) s_warp[warp] = wsum;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned int tot = 0;
        for (int w = 0; w < kFinThreads / 32; ++w) tot += s_warp[w];
        s_total = tot;
        unsigned long long base = 0;
        if (tot > 0) {
            base = atomicAdd(p.cursor, (unsigned long long)tot);
            if (base + tot > p.arena_cap) {
                *p.overflow = 1;
                tot = 0;
                s_total = 0;
            }
        }
        s_base = base;
        p.pair_cnt[pair] = (int32_t)tot;
        p.pair_off[pair] = base;
    }
    __syncthreads();
    if (s_total == 0) return;

    // pass 2: stable compaction in ascending query index (rows were written by this block: visible after the barrier)
    unsigned long long running = s_base;
    for (int q0 = 0; q0 < fq; q0 += kFinThreads) {
        const int q = q0 + threadIdx.x;
        const u64 v = (q < fq) ? rk1[q] : kKeyInit;
        const bool keep = v != kKeyInit;
        const unsigned int bal = __ballot_sync(0xffffffffu, keep);
        __syncthreads();  // s_warp reuse
        if (lane == 0) s_warp[warp] = __popc(bal);
        __syncthreads();
        unsigned int before = 0, total = 0;
#pragma unroll
        for (int w = 0; w < kFinThreads / 32; ++w) {
            const unsigned int c = s_warp[w];
            before += (w < warp) ? c : 0u;
            total += c;
        }
        if (keep) {
            esfm_dmatch_t m;
            m.queryIdx = q;
            m.trainIdx = (int32_t)(uint32_t)v;
            m.imgIdx = 0;
            m.distance = __uint_as_float((uint32_t)(v >> 32));
            p.arena[running + before + __popc(bal & ((1u << lane) - 1u))] = m;
        }
        running += total;
    }
}

// SURF fast sweep -> which rows need the exact fallback sweep, from the sweep's values alone (no descriptor reads): every row that
// eval_rows_win could not decide on its values (win_ratio_class == 2), and with ratio = inf every row whose nearest column is not
// certain (s2 - s1 <= 2 e).  Their indices go on the pair's gather list, any order (the fallback sweep writes back by row index).
__global__ void __launch_bounds__(kFinThreads) win_classify_kernel(const FinalizeParams p) {
    const int pair = blockIdx.x;
    const PairDesc pd = p.pairs[pair];
    const int fq = p.frame_rows[pd.q_frame], ft = p.frame_rows[pd.t_frame];
    const bool no_ratio = p.ratio == __longlong_as_double(0x7ff0000000000000LL);
    __shared__ unsigned int s_cnt;
    if (threadIdx.x == 0) s_cnt = 0;
    __syncthreads();
    if (fq > 0 && ft >= (no_ratio ? 1 : 2) && (no_ratio || p.ratio > 0.0)) {      // (else finalize emits nothing for the pair)
        const u64* rk1 = p.keys + (size_t)pair * 4 * p.stride;
        const u64* rk2 = rk1 + p.stride;
        const float* row_eps = p.row_eps + p.frame_row_off[pd.q_frame];
        const float nq = p.frame_norm[pd.q_frame], nt = p.frame_norm[pd.t_frame];
        const float r2 = (float)(p.ratio * p.ratio);
        int* gl = p.gather + (size_t)pair * p.stride;
        for (int q = threadIdx.x; q < fq; q += kFinThreads) {
            const u64 k1 = rk1[q], k2 = rk2[q];
            if (k1 == kKeyInit) continue;                             // no column at all
            // no second chain: s2 = +inf, settled -- the best chain holds every column, and finalize evaluates it exactly
            const float s1 = __uint_as_float((uint32_t)(k1 >> 32));
            const float s2 = k2 == kKeyInit ? __int_as_float(0x7f800000) : __uint_as_float((uint32_t)(k2 >> 32));
            const float e = win_fast_eps(row_eps[q], nq, nt);
            const bool unsettled = no_ratio ? !(s2 - s1 > 2.f * e) : win_ratio_class(s1, s2, e, r2) == 2;
            if (unsettled) gl[atomicAdd(&s_cnt, 1u)] = q;
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        p.gather_cnt[pair] = (int)s_cnt;
        if (s_cnt) atomicAdd(p.fallback_rows, (unsigned long long)s_cnt);
    }
}

}  // namespace

cudaError_t launch_win_classify(const FinalizeParams& p, cudaStream_t s) {
    if (p.n_pairs <= 0) return cudaSuccess;
    win_classify_kernel<<<p.n_pairs, kFinThreads, 0, s>>>(p);
    return cudaGetLastError();
}

cudaError_t launch_finalize(const FinalizeParams& p, cudaStream_t s) {
    if (p.n_pairs <= 0) return cudaSuccess;
    if (p.kind == ESFM_KIND_F32X64) finalize_kernel<ESFM_KIND_F32X64><<<p.n_pairs, kFinThreads, 0, s>>>(p);
    else finalize_kernel<ESFM_KIND_B256><<<p.n_pairs, kFinThreads, 0, s>>>(p);
    return cudaGetLastError();
}

}  // namespace esfm
