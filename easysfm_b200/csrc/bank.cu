// bank.cu -- derived device layouts of the descriptor bank (run once per esfm_bank_commit).
//
// F32X64: rows_f32[total_rows][64] (row-major, as the reference's cv::Mat holds SURF descriptors,
// cpp_code/include/utility.h:31) -> k-major 128-row tiles + half squared norms, the operand layout the
// sweep kernel bulk-copies into shared memory with one cp.async.bulk per tile.
#include "tc_layout.cuh"

namespace esfm {

__global__ void __launch_bounds__(256) pack_f32_kernel(const float* __restrict__ rows, const int* __restrict__ frame_rows,
                                                       const int* __restrict__ frame_row_off,
                                                       const int* __restrict__ frame_tile_off, int n_frames,
                                                       float* __restrict__ kmajor) {
    __shared__ float tile[kTile][kDim + 1];
    const int t = blockIdx.x;
    // frame owning tile t: last f with frame_tile_off[f] <= t
    int lo = 0, hi = n_frames - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (frame_tile_off[mid] <= t) lo = mid; else hi = mid - 1;
    }
    const int f = lo;
    const int row0 = (t - frame_tile_off[f]) * kTile;
    int valid = frame_rows[f] - row0;
    valid = valid < 0 ? 0 : (valid > kTile ? kTile : valid);
    const float4* src = reinterpret_cast<const float4*>(rows + ((size_t)frame_row_off[f] + row0) * kDim);
    for (int idx = threadIdx.x; idx < kTile * (kDim / 4); idx += blockDim.x) {
        const int r = idx / (kDim / 4), c4 = idx % (kDim / 4);
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (r < valid) v = src[(size_t)r * (kDim / 4) + c4];
        tile[r][c4 * 4 + 0] = v.x;
        tile[r][c4 * 4 + 1] = v.y;
        tile[r][c4 * 4 + 2] = v.z;
        tile[r][c4 * 4 + 3] = v.w;
    }
    __syncthreads();
    float* out = kmajor + (size_t)t * kTileFloats;
    for (int idx = threadIdx.x; idx < kDim * kTile; idx += blockDim.x) {
        const int k = idx / kTile, r = idx % kTile;
        out[idx] = tile[r][k];
    }
    if (threadIdx.x < kTile) {
        const int r = threadIdx.x;
        float s = 0.f;
#pragma unroll 8
        for (int k = 0; k < kDim; ++k) s = __fmaf_rn(tile[r][k], tile[r][k], s);
        // pad rows: +inf half-norm makes every distance involving them +inf, so they never pass a threshold
        out[kDim * kTile + r] = (r < valid) ? 0.5f * s : __int_as_float(0x7f800000);
    }
}

cudaError_t launch_pack_f32(const float* rows, const int* frame_rows, const int* frame_row_off, const int* frame_tile_off,
                            int n_frames, int n_tiles_total, float* kmajor, cudaStream_t s) {
    if (n_tiles_total <= 0) return cudaSuccess;
    pack_f32_kernel<<<n_tiles_total, 256, 0, s>>>(rows, frame_rows, frame_row_off, frame_tile_off, n_frames, kmajor);
    return cudaGetLastError();
}

// F32X64 -> the tensor-core operand images of tc_layout.cuh: per 128-row tile one contiguous 69632-byte image = 16 groups
// x 4096 B of SWIZZLE_128B hi/lo atoms + 16 x 256 B of augmented (train-role) columns.  One block per tile; byte-for-byte
// what tc_pack_row_host(query_role = false) writes.
__global__ void __launch_bounds__(256) pack_tc_kernel(const float* __restrict__ rows, const int* __restrict__ frame_rows,
                                                      const int* __restrict__ frame_row_off,
                                                      const int* __restrict__ frame_tile_off, int n_frames,
                                                      unsigned char* __restrict__ tc_main) {
    __shared__ float tile[kTile][kDim + 4];
    const int t = blockIdx.x;
    int lo = 0, hi = n_frames - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (frame_tile_off[mid] <= t) lo = mid; else hi = mid - 1;
    }
    const int f = lo;
    const int row0 = (t - frame_tile_off[f]) * kTile;
    int valid = frame_rows[f] - row0;
    valid = valid < 0 ? 0 : (valid > kTile ? kTile : valid);
    const float4* src = reinterpret_cast<const float4*>(rows + ((size_t)frame_row_off[f] + row0) * kDim);
    unsigned char* out = tc_main + (size_t)t * kTcTileBytes;
    for (int idx = threadIdx.x; idx < kTile * (kDim / 4); idx += blockDim.x) {
        const int r = idx / (kDim / 4), c4 = idx % (kDim / 4);
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (r < valid) v = src[(size_t)r * (kDim / 4) + c4];
        *reinterpret_cast<float4*>(&tile[r][c4 * 4]) = v;
        const float4 h = make_float4(tc_tf32_hi(v.x), tc_tf32_hi(v.y), tc_tf32_hi(v.z), tc_tf32_hi(v.w));
        const float4 l = make_float4(v.x - h.x, v.y - h.y, v.z - h.z, v.w - h.w);
        const int k = c4 * 4;
        const int off = (r >> 3) * kTcGroupBytes + (k >> 5) * 1024 + tc_sw128_off(r & 7, k & 31);
        *reinterpret_cast<float4*>(out + off) = h;
        *reinterpret_cast<float4*>(out + off + 2048) = l;
    }
    __syncthreads();
    if (threadIdx.x < kTile) {
        const int r = threadIdx.x;
        float s = 0.f;
#pragma unroll 8
        for (int k = 0; k < kDim; ++k) s = __fmaf_rn(tile[r][k], tile[r][k], s);
        const float h = (r < valid) ? 0.5f * s : kTcPadNorm;
        float hh, hm, hl;
        tc_split3(h, hh, hm, hl);
        // train role: (-h_h, -h_m, -h_l, -1 | -1, -1, 0, 0) against the query's (1, 1, 1, hq_h | hq_m, hq_l, 0, 0)
        unsigned char* a = out + kTcMainBytes + (r >> 3) * kTcAugGroupBytes + (r & 7) * 16;
        *reinterpret_cast<float4*>(a) = make_float4(-hh, -hm, -hl, -1.f);
        *reinterpret_cast<float4*>(a + 128) = make_float4(-1.f, -1.f, 0.f, 0.f);
    }
}

cudaError_t launch_pack_tc(const float* rows, const int* frame_rows, const int* frame_row_off, const int* frame_tile_off,
                           int n_frames, int n_tiles_total, unsigned char* tc_main, cudaStream_t s) {
    if (n_tiles_total <= 0) return cudaSuccess;
    pack_tc_kernel<<<n_tiles_total, 256, 0, s>>>(rows, frame_rows, frame_row_off, frame_tile_off, n_frames, tc_main);
    return cudaGetLastError();
}

// F32X64 -> the 16-bit split ("H") images of tc_layout.cuh for sweep_win.cu: per 128-row tile 16 groups x 2048 B = [a k0..63][b k0..63]
// SWIZZLE_128B atoms of fp16 (a = fp16(x), b = fp16(x - a)) + the same 16 x 256 B augmented TF32 columns as the 3xTF32 image.
// One block per tile, one thread per (row, 8 dims = one 16-byte chunk of each atom); byte-for-byte tch_pack_row_host.
// Also the two inputs of win_fast_eps: per row |x - fp16(x)|_2 (the rounding of the sweep's query writers) and per frame the largest
// |x|_2 (frame_norm must be zero on entry), both rounded up.
__global__ void __launch_bounds__(256) pack_tch_kernel(const float* __restrict__ rows, const int* __restrict__ frame_rows,
                                                       const int* __restrict__ frame_row_off,
                                                       const int* __restrict__ frame_tile_off, int n_frames,
                                                       unsigned char* __restrict__ tc_main, float* __restrict__ row_eps,
                                                       float* __restrict__ frame_norm) {
    __shared__ float tile[kTile][kDim + 4];
    const int t = blockIdx.x;
    int lo = 0, hi = n_frames - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (frame_tile_off[mid] <= t) lo = mid; else hi = mid - 1;
    }
    const int f = lo;
    const int row0 = (t - frame_tile_off[f]) * kTile;
    int valid = frame_rows[f] - row0;
    valid = valid < 0 ? 0 : (valid > kTile ? kTile : valid);
    const float4* src = reinterpret_cast<const float4*>(rows + ((size_t)frame_row_off[f] + row0) * kDim);
    unsigned char* out = tc_main + (size_t)t * kTchTileBytes;
    for (int idx = threadIdx.x; idx < kTile * (kDim / 8); idx += blockDim.x) {
        const int r = idx / (kDim / 8), c8 = idx % (kDim / 8);
        float4 v0 = make_float4(0.f, 0.f, 0.f, 0.f), v1 = v0;
        if (r < valid) { v0 = src[(size_t)r * (kDim / 4) + 2 * c8]; v1 = src[(size_t)r * (kDim / 4) + 2 * c8 + 1]; }
        *reinterpret_cast<float4*>(&tile[r][c8 * 8]) = v0;
        *reinterpret_cast<float4*>(&tile[r][c8 * 8 + 4]) = v1;
        const float xs[8] = {v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w};
        uint32_t a[8], b[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            a[j] = tch_f2h(xs[j]);
            b[j] = tch_f2h(xs[j] - tch_h2f(a[j]));
        }
        const int off = (r >> 3) * kTchGroupBytes + tch_sw128_off(r & 7, c8 * 8);
        *reinterpret_cast<uint4*>(out + off) = make_uint4(a[0] | (a[1] << 16), a[2] | (a[3] << 16), a[4] | (a[5] << 16), a[6] | (a[7] << 16));
        *reinterpret_cast<uint4*>(out + off + 1024) = make_uint4(b[0] | (b[1] << 16), b[2] | (b[3] << 16), b[4] | (b[5] << 16), b[6] | (b[7] << 16));
    }
    __syncthreads();
    if (threadIdx.x < kTile) {
        const int r = threadIdx.x;
        float s = 0.f, se = 0.f;
#pragma unroll 8
        for (int k = 0; k < kDim; ++k) {
            const float x = tile[r][k], d = x - tch_h2f(tch_f2h(x));     // exact in fp32
            s = __fmaf_rn(x, x, s);
            se = __fmaf_rn(d, d, se);
        }
        if (r < valid) {
            // (64 fused steps: relative error < 2^-18 on the sums, the square roots are rounded up)
            row_eps[frame_row_off[f] + row0 + r] = __fsqrt_ru(se) * (1.f + 0x1p-16f);
            atomicMax(reinterpret_cast<int*>(frame_norm + f), __float_as_int(__fsqrt_ru(s) * (1.f + 0x1p-16f)));
        }
        const float h = (r < valid) ? 0.5f * s : kTcPadNorm;
        float hh, hm, hl;
        tc_split3(h, hh, hm, hl);
        unsigned char* a = out + kTchMainBytes + (r >> 3) * kTcAugGroupBytes + (r & 7) * 16;
        *reinterpret_cast<float4*>(a) = make_float4(-hh, -hm, -hl, -1.f);
        *reinterpret_cast<float4*>(a + 128) = make_float4(-1.f, -1.f, 0.f, 0.f);
    }
}

cudaError_t launch_pack_tch(const float* rows, const int* frame_rows, const int* frame_row_off, const int* frame_tile_off,
                            int n_frames, int n_tiles_total, unsigned char* tc_main, float* row_eps, float* frame_norm, cudaStream_t s) {
    if (n_tiles_total <= 0) return cudaSuccess;
    cudaError_t e = cudaMemsetAsync(frame_norm, 0, (size_t)n_frames * sizeof(float), s);
    if (e != cudaSuccess) return e;
    pack_tch_kernel<<<n_tiles_total, 256, 0, s>>>(rows, frame_rows, frame_row_off, frame_tile_off, n_frames, tc_main, row_eps, frame_norm);
    return cudaGetLastError();
}

// F32X64 input range (esfm_bank_commit): per frame the largest |x| of any component, as float bits with the sign dropped (the integer
// order of non-negative floats is their numeric order, so atomicMax works on them); an inf or NaN component leaves bits >= 0x7f800000.
// One block per 128-row tile, one atomic per tile; frame_absmax must be zero on entry.
__global__ void __launch_bounds__(256) frame_absmax_kernel(const float* __restrict__ rows, const int* __restrict__ frame_rows,
                                                           const int* __restrict__ frame_row_off, const int* __restrict__ frame_tile_off,
                                                           int n_frames, unsigned* __restrict__ frame_absmax) {
    const int t = blockIdx.x;
    int lo = 0, hi = n_frames - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (frame_tile_off[mid] <= t) lo = mid; else hi = mid - 1;
    }
    const int f = lo;
    const int row0 = (t - frame_tile_off[f]) * kTile;
    int valid = frame_rows[f] - row0;
    valid = valid < 0 ? 0 : (valid > kTile ? kTile : valid);
    const float4* src = reinterpret_cast<const float4*>(rows + ((size_t)frame_row_off[f] + row0) * kDim);
    unsigned m = 0;
    for (int idx = threadIdx.x; idx < valid * (kDim / 4); idx += blockDim.x) {
        const float4 v = src[idx];
        m = max(m, max(max(__float_as_uint(v.x) & 0x7fffffffu, __float_as_uint(v.y) & 0x7fffffffu),
                       max(__float_as_uint(v.z) & 0x7fffffffu, __float_as_uint(v.w) & 0x7fffffffu)));
    }
    m = __reduce_max_sync(0xffffffffu, m);
    __shared__ unsigned warp_max[8];
    if ((threadIdx.x & 31) == 0) warp_max[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 8; ++w) m = max(m, warp_max[w]);
        if (m) atomicMax(frame_absmax + f, m);
    }
}

cudaError_t launch_frame_absmax(const float* rows, const int* frame_rows, const int* frame_row_off, const int* frame_tile_off, int n_frames,
                                int n_tiles_total, unsigned* frame_absmax, cudaStream_t s) {
    cudaError_t e = cudaMemsetAsync(frame_absmax, 0, (size_t)n_frames * sizeof(unsigned), s);
    if (e != cudaSuccess || n_tiles_total <= 0) return e;
    frame_absmax_kernel<<<n_tiles_total, 256, 0, s>>>(rows, frame_rows, frame_row_off, frame_tile_off, n_frames, frame_absmax);
    return cudaGetLastError();
}

// B256 -> the FP8 tile images of tc_layout.cuh (Hamming on the tensor cores): one block per 128-row tile, one thread per
// (row, 32-bit word): 32 bits -> 32 bytes of +-1.0 (E4M3), written as two 16-byte chunks into the SWIZZLE_128B atoms.
__global__ void __launch_bounds__(256) pack_tc8_kernel(const uint32_t* __restrict__ rows, const int* __restrict__ frame_rows,
                                                       const int* __restrict__ frame_row_off,
                                                       const int* __restrict__ frame_tile_off, int n_frames,
                                                       unsigned char* __restrict__ tc_main, int z_mode) {
    const int t = blockIdx.x;
    int lo = 0, hi = n_frames - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (frame_tile_off[mid] <= t) lo = mid; else hi = mid - 1;
    }
    const int f = lo;
    const int row0 = (t - frame_tile_off[f]) * kTile;
    int valid = frame_rows[f] - row0;
    valid = valid < 0 ? 0 : (valid > kTile ? kTile : valid);
    const uint32_t* src = rows + ((size_t)frame_row_off[f] + row0) * 8;
    unsigned char* out = tc_main + (size_t)t * kTc8TileBytes;
    for (int idx = threadIdx.x; idx < kTile * 8; idx += blockDim.x) {
        const int r = idx >> 3, w = idx & 7;                   // row, word: bits 32 w .. 32 w + 31 = elements k
        uint4 c0 = make_uint4(0u, 0u, 0u, 0u), c1 = c0;          // pad rows: all-zero operands (+0.0)
        if (r < valid) {
            const uint32_t x = src[(size_t)r * 8 + w];
            if (z_mode) {     // "Z" encoding (tc_layout.cuh): bit 0 -> -64, bit 1 -> +64
                c0 = make_uint4(tcz_expand4_t(x), tcz_expand4_t(x >> 4), tcz_expand4_t(x >> 8), tcz_expand4_t(x >> 12));
                c1 = make_uint4(tcz_expand4_t(x >> 16), tcz_expand4_t(x >> 20), tcz_expand4_t(x >> 24), tcz_expand4_t(x >> 28));
            } else {
                c0 = make_uint4(tc8_expand4(x), tc8_expand4(x >> 4), tc8_expand4(x >> 8), tc8_expand4(x >> 12));
                c1 = make_uint4(tc8_expand4(x >> 16), tc8_expand4(x >> 20), tc8_expand4(x >> 24), tc8_expand4(x >> 28));
            }
        }
        const int k = w * 32;                                   // first element of this word
        unsigned char* atom = out + (r >> 3) * kTc8GroupBytes + (k >> 7) * 1024;
        *reinterpret_cast<uint4*>(atom + tc8_sw128_off(r & 7, k & 127)) = c0;
        *reinterpret_cast<uint4*>(atom + tc8_sw128_off(r & 7, (k & 127) + 16)) = c1;
    }
    if (threadIdx.x < kTile) {
        const int r = threadIdx.x;
        // train role: (-448, tpad ? -448 : 0, -16, 0 ...) against the query's (qpad ? 448 : 0, 448, 16, 0 ...)
        unsigned char* a = out + kTc8MainBytes + (r >> 3) * kTcAugGroupBytes + (r & 7) * 16;
        if (z_mode) {
            // offset slots + the row's index inside its frame, digit by digit; pad rows stay all-zero (masked by index in the sweep)
            uint32_t w[8] = {0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u};
            if (r < valid) tcz_train_aug((uint32_t)(row0 + r), w);
            *reinterpret_cast<uint4*>(a) = make_uint4(w[0], w[1], w[2], w[3]);
            *reinterpret_cast<uint4*>(a + 128) = make_uint4(w[4], w[5], w[6], w[7]);
        } else {
        *reinterpret_cast<uint4*>(a) = make_uint4(kFp8Neg448 | ((r < valid ? 0u : kFp8Neg448) << 8) | (kFp8Neg16 << 16), 0u, 0u, 0u);
        *reinterpret_cast<uint4*>(a + 128) = make_uint4(0u, 0u, 0u, 0u);
        }
    }
}

cudaError_t launch_pack_tc8(const uint32_t* rows, const int* frame_rows, const int* frame_row_off, const int* frame_tile_off,
                            int n_frames, int n_tiles_total, unsigned char* tc_main, int z_mode, cudaStream_t s) {
    if (n_tiles_total <= 0) return cudaSuccess;
    pack_tc8_kernel<<<n_tiles_total, 256, 0, s>>>(rows, frame_rows, frame_row_off, frame_tile_off, n_frames, tc_main, z_mode);
    return cudaGetLastError();
}

}  // namespace esfm
