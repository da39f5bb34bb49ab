// tc_sweep_common.cuh -- what the tensor-core sweep kernels (sweep_l2_tc.cu: 3xTF32 / FP8 "Z"; sweep_win.cu: 16-bit split / FP16
// accumulators with window keys) share: the role layout of the 24-warp CTA, barrier waits with a deadlock watchdog, work decoding,
// and the column-event handlers (packed (value, query row) keys posted with fire-and-forget atomics).
#pragma once
#include "tc_layout.cuh"

namespace esfm {
namespace {

constexpr int kTcColParts = 4;                          // column quarters of a train tile, one per epilogue warp of a lane quarter
constexpr int kTcEpiWarps = 4 * kTcColParts;            // 16 epilogue warps: enough to hide the epilogue's dependent-issue latency
constexpr int kTcEpiThreads = kTcEpiWarps * 32;
constexpr int kTcThreads = kTcEpiThreads + 256;         // + 2 service warpgroups: TMA producer, MMA issuer, (2 idle), 4 query writers
constexpr int kTcWriterWarp0 = kTcEpiWarps + 4;         // warps 20..23: warp % 4 covers the four TMEM lane quarters
// setmaxnreg works on whole warpgroups: the kernel launches at 80 registers/thread (768 threads), the two service
// warpgroups shrink to 40 and the four epilogue warpgroups grow to 96 (32 accumulator columns + 8 group maxima + thresholds
// live at once).  setmaxnreg.inc can only take what setmaxnreg.dec of the SAME CTA released (the unallocated rest of the
// register file is not in the pool -- asking for more blocks forever), hence the balance check.
constexpr int kTcLaunchRegs = 80, kTcEpiRegs = 96, kTcServiceRegs = 48;
static_assert(256 * (kTcLaunchRegs - kTcServiceRegs) >= kTcEpiThreads * (kTcEpiRegs - kTcLaunchRegs), "setmaxnreg pool would deadlock");
static_assert(kTcThreads * kTcLaunchRegs <= 65536 && (65536 / kTcThreads) / 8 * 8 == kTcLaunchRegs, "launch register count drifted");
constexpr int kTcPartCols = kTile / kTcColParts;        // 32 columns per epilogue thread and stage
constexpr int kTcStages = 3;                 // shared-memory train stages (68 KB each)
constexpr int kTcThrBytes = kTile * 4;                  // 512: column thresholds riding with a train tile
constexpr int kTcThrStages = 4;                         // threshold snapshots have their own (deeper) ring

struct TcUnit {
    int pair, q_frame, t_frame;
    int nqt, ntt;
    int qb0, qb1;        // query TILES [qb0, qb1) of this unit
};

__device__ __forceinline__ TcUnit tc_decode_unit(const SweepParams& p, int unit) {
    TcUnit u;
    u.pair = unit / p.units_per_pair;
    const int part = unit - u.pair * p.units_per_pair;
    const PairDesc pd = p.pairs[u.pair];
    u.q_frame = pd.q_frame;
    u.t_frame = pd.t_frame;
    u.nqt = p.frame_tile_off[pd.q_frame + 1] - p.frame_tile_off[pd.q_frame];
    u.ntt = p.frame_tile_off[pd.t_frame + 1] - p.frame_tile_off[pd.t_frame];
    u.qb0 = (int)((long long)u.nqt * part / p.units_per_pair);
    u.qb1 = (int)((long long)u.nqt * (part + 1) / p.units_per_pair);
    if (p.frame_rows[pd.t_frame] < 1) u.qb1 = u.qb0;
    return u;
}

// Watchdog of every barrier wait: 4 s on one barrier is certainly a pipeline deadlock; trap, so that it surfaces as a launch
// failure instead of a hung GPU (the wall clock is only read every 1024 polls).
__device__ __forceinline__ void tc_watchdog(uint32_t& polls, unsigned long long& t0) {
    if ((++polls & 0x3ffu) == 0) {
        unsigned long long now;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
        if (t0 == 0) t0 = now;
        else if (now - t0 > 4000000000ull) __trap();
    }
}

struct RowTop2 {
    float v1, v2;        // 1/2 d^2 of the best / second best so far
    uint32_t i1, i2;
};

// Barrier waits.  Every waiting warp shares an SM sub-partition with four epilogue warps, and a polling loop is not free:
// with try_wait + 40 ns sleeps the six service warps and the parked epilogue warps together executed > 40 % of all
// instructions of the kernel (ncu source page), taken from the issue slots of the warps that had work.  (The suspend-time
// hint of try_wait does not park a warp for anything near the hinted time.)  So every role sleeps between polls for as long
// as its place in the pipeline tolerates: SLEEP_NS is a template argument.
__device__ __forceinline__ void named_bar_sync(int id, int threads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(threads) : "memory"); }
__device__ __forceinline__ void named_bar_arrive(int id, int threads) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(threads) : "memory"); }

template <int SLEEP_NS>
__device__ __forceinline__ void mbar_wait_sleep(uint64_t* bar, uint32_t parity) {
    uint32_t ok = 0, polls = 0;
    unsigned long long t0 = 0;
    while (true) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok)
            : "r"(smem_u32(bar)), "r"(parity)
            : "memory");
        if (ok) break;
        if (SLEEP_NS > 0) __nanosleep(SLEEP_NS);
        tc_watchdog(polls, t0);
    }
}
// Measured: sleeping 60-200 ns in the producer / issuer / epilogue waits costs 3 % (wake-up latency sits on the pipeline's
// critical path), so those keep polling; the four writer warps do not poll at all (named barrier, see below).
constexpr int kTcSleepProducer = 40;
constexpr int kTcSleepIssuer = 40;
constexpr int kTcSleepEpilogue = 0;

constexpr int kTcScCols = 4;                                   // columns staged per column-event round (a group of 4 accumulator columns)
constexpr int kTcScBytes = kTcEpiWarps * kTcScCols * 32 * 4;   // 8 KB: per epilogue warp [4 columns][32 lanes] floats

// Column events of one group of 4 train columns, for the whole warp: ONE compact body, never inlined.  The selection epilogue
// holds a query row's 32 accumulators in registers, which can only be indexed statically -- so every earlier event handler was
// either unrolled per column (19 KB of rarely executed code: instruction-cache misses showed up as 15 % "no instruction" stalls)
// or dug the value out of the registers with select trees and elected a winner per column in a serial loop (~70 instructions
// and ~300 cycles of dependent latency PER EVENT; the first query block of a pair, where every column gets its first minimum,
// ran 10x slower than the others and held 60 % of all events).  Here the caller parks the group's 4 x 32 candidate keys in a
// per-warp shared-memory scratch (4 STS) and the warp reduces all four columns AT ONCE: 8 lanes per column, each takes 4 rows
// (one LDS.128), then three xor-shuffle rounds of (key, row) pairs -- lowest key, lowest query row on ties -- and the 4 leader
// lanes post their column's winner with two fire-and-forget atomics (packed key; threshold) if it beats the threshold.
// ~45 instructions per group whatever the number of events in it.
// Keys are "smaller = nearer" non-negative floats: the Z key itself, else max(1/2 d^2, 0) (or 2 x hamming).
// Scratch and thresholds are 32-bit shared-window addresses (generic pointers cost a dozen 64-bit instructions per call).
// One column's event posted by the lane itself, branch-free: if (ok && y <= t) { RED.MIN.64 ck[j] <- (y bits, qrow); RED.MIN.32
// tau[j] <- bits(y - thr_sub) }.  Inline PTX because the compiler turns the C++ form into a branch per column (BSSY / BRA /
// BSYNC + re-derived addresses: ~25 instructions and one more serialised decision point each); here it is 6 predicated
// instructions with the column offset as an immediate.
template <int J>
__device__ __forceinline__ void tc_col_post(float y, float t, int ok, u64* ck, uint32_t* tau, uint32_t qrow, float thr_sub) {
    asm volatile(
        "{\n\t.reg .pred p, q;\n\t.reg .b64 k;\n\t.reg .f32 s;\n\t.reg .b32 yb, sb;\n\t"
        "setp.ne.s32 q, %2, 0;\n\t"
        "setp.le.and.f32 p, %0, %1, q;\n\t"
        "mov.b32 yb, %0;\n\t"
        "mov.b64 k, {%5, yb};\n\t"
        "sub.f32 s, %0, %6;\n\t"
        "mov.b32 sb, s;\n\t"
        "@p red.global.min.u64 [%3 + %7], k;\n\t"
        "@p red.global.min.u32 [%4 + %8], sb;\n\t}"
        ::"f"(y), "f"(t), "r"(ok), "l"(ck), "l"(tau), "r"(qrow), "f"(thr_sub), "n"(J * 8), "n"(J * 4)
        : "memory");
}

template <bool kZ>
__device__ __noinline__ void tc_col_group(uint32_t sc_addr, uint32_t thr_addr, u64* ck, uint32_t* tau, uint32_t qrow0, float thr_sub, int dbg) {
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t col = lane >> 3, r4 = (lane & 7u) * 4u;
    float y0, y1, y2, y3, t;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(y0), "=f"(y1), "=f"(y2), "=f"(y3) : "r"(sc_addr + col * 128u + r4 * 4u));
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(t) : "r"(thr_addr + col * 4u));
    float best = y0;
    uint32_t br = r4;
    if (y1 < best) { best = y1; br = r4 + 1; }
    if (y2 < best) { best = y2; br = r4 + 2; }
    if (y3 < best) { best = y3; br = r4 + 3; }
#pragma unroll
    for (int d = 1; d <= 4; d <<= 1) {
        const float oy = __shfl_xor_sync(0xffffffffu, best, d);
        const uint32_t orow = __shfl_xor_sync(0xffffffffu, br, d);
        const bool take = oy < best || (oy == best && orow < br);
        best = take ? oy : best;
        br = take ? orow : br;
    }
    if ((lane & 7u) == 0 && best <= t && !(dbg & 32)) {
        const uint32_t bits = __float_as_uint(best);
        atomicMin(ck + col, make_key(bits, qrow0 + br));
        atomicMin(tau + col, kZ ? __float_as_uint(best - thr_sub) : bits);
    }
}

}  // namespace
}  // namespace esfm
