// capi.cu -- host side of libesfm_match.so: the single-device part of the C ABI declared in include/esfm_match.h
// (multi.cu holds esfm_multi_*).
//
// Host logic only (bank staging, pair-batch chunking, scratch management, result bookkeeping); every distance, selection,
// ratio, cross-check and compaction step runs in the CUDA kernels of this library.  There is no CPU fallback: if the
// device or a kernel fails the call fails.
#include <sys/mman.h>

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <new>

#include "host_internal.h"

using namespace esfm;

// ------------------------------------------------------------------------------------------------
// error plumbing
// ------------------------------------------------------------------------------------------------
namespace esfm {

thread_local std::string g_last_error;

int fail(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_last_error = buf;
    return code;
}

// ------------------------------------------------------------------------------------------------
// helper threads for large host copies
// ------------------------------------------------------------------------------------------------
CopyPool::CopyPool(int helpers) {
    jobs_.resize((size_t)helpers);
    for (int k = 0; k < helpers; ++k) threads_.emplace_back(&CopyPool::worker, this, k);
}

CopyPool::~CopyPool() {
    {
        std::lock_guard<std::mutex> lk(mu_);
        stop_ = true;
        ++epoch_;
    }
    cv_work_.notify_all();
    for (auto& t : threads_) t.join();
}

void CopyPool::worker(int k) {
    uint64_t seen = 0;
    for (;;) {
        Job j;
        {
            std::unique_lock<std::mutex> lk(mu_);
            cv_work_.wait(lk, [&] { return epoch_ != seen; });
            seen = epoch_;
            if (stop_) return;
            j = jobs_[(size_t)k];
        }
        if (j.bytes) memcpy(j.dst, j.src, j.bytes);
        {
            std::lock_guard<std::mutex> lk(mu_);
            if (--pending_ == 0) cv_done_.notify_one();
        }
    }
}

void CopyPool::copy(void* dst, const void* src, size_t bytes) {
    const size_t parts = threads_.size() + 1;
    if (bytes < ((size_t)1 << 20) || threads_.empty()) {
        if (bytes) memcpy(dst, src, bytes);
        return;
    }
    const size_t slice = ((bytes / parts) + 4095) & ~(size_t)4095;
    {
        std::lock_guard<std::mutex> lk(mu_);
        for (size_t k = 0; k < threads_.size(); ++k) {
            const size_t off = std::min(bytes, (k + 1) * slice), end = std::min(bytes, (k + 2) * slice);
            jobs_[k] = Job{(char*)dst + off, (const char*)src + off, end - off};
        }
        pending_ = (int)threads_.size();
        ++epoch_;
    }
    cv_work_.notify_all();
    memcpy(dst, src, std::min(bytes, slice));   // the calling thread takes the first slice
    std::unique_lock<std::mutex> lk(mu_);
    cv_done_.wait(lk, [&] { return pending_ == 0; });
}

// ------------------------------------------------------------------------------------------------
// pinned buffer pool, heap segments, digests
// ------------------------------------------------------------------------------------------------
void* pool_acquire(esfm_ctx* ctx, size_t bytes, size_t* got) {
    size_t best = (size_t)-1;
    for (size_t i = 0; i < ctx->pool.size(); ++i)
        if (!ctx->pool[i].in_use && ctx->pool[i].bytes >= bytes && (best == (size_t)-1 || ctx->pool[i].bytes < ctx->pool[best].bytes)) best = i;
    if (best != (size_t)-1) {
        ctx->pool[best].in_use = true;
        if (got) *got = ctx->pool[best].bytes;
        return ctx->pool[best].ptr;
    }
    // drop idle buffers that were too small, then allocate with 25% headroom
    for (size_t i = 0; i < ctx->pool.size();) {
        if (!ctx->pool[i].in_use) { cudaFreeHost(ctx->pool[i].ptr); ctx->pool.erase(ctx->pool.begin() + i); } else ++i;
    }
    size_t want = bytes + bytes / 4 + 4096;
    void* p = nullptr;
    if (cudaMallocHost(&p, want) != cudaSuccess) {
        cudaGetLastError();
        want = bytes;
        if (cudaMallocHost(&p, want) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    }
    ctx->pool.push_back({p, want, true});
    if (got) *got = want;
    return p;
}

void pool_release(esfm_ctx* ctx, void* ptr) {
    if (!ptr || !ctx) return;
    for (auto& b : ctx->pool)
        if (b.ptr == ptr) { b.in_use = false; return; }
}

// Pageable storage of a multi-chunk batch's matches: 2 MB aligned and advised as huge pages, so that first-touching
// gigabytes of it from several worker threads is a few thousand page faults, not millions.
esfm_dmatch_t* heap_segment_alloc(size_t n_matches) {
    const size_t bytes = std::max<size_t>(n_matches * sizeof(esfm_dmatch_t), 16);
    void* p = nullptr;
    if (bytes >= ((size_t)4 << 20)) {
        if (posix_memalign(&p, (size_t)2 << 20, bytes) != 0) return nullptr;
        madvise(p, bytes, MADV_HUGEPAGE);
    } else {
        p = malloc(bytes);
    }
    return (esfm_dmatch_t*)p;
}

// 64-bit digest of one pair's matches: count, then every record's indices and distance bits weighted by its position
// (order-sensitive, so a permuted output does not pass; sums commute, so the loop vectorises).
uint64_t digest_matches(const esfm_dmatch_t* m, int n) {
    uint64_t h = 0x9E3779B97F4A7C15ull * (uint64_t)(n + 1);
    for (int i = 0; i < n; ++i) {
        uint32_t db;
        memcpy(&db, &m[i].distance, 4);
        const uint64_t rec = ((uint64_t)(uint32_t)m[i].queryIdx * 0xD6E8FEB86659FD93ull) ^ ((uint64_t)(uint32_t)m[i].trainIdx * 0xA0761D6478BD642Full) ^
                             ((uint64_t)db * 0xE7037ED1A0B428DBull) ^ ((uint64_t)(uint32_t)m[i].imgIdx << 17);
        h += rec * (uint64_t)(2 * i + 1);
    }
    return h;
}

}  // namespace esfm

// ------------------------------------------------------------------------------------------------
// small helpers
// ------------------------------------------------------------------------------------------------
int esfm::set_device(esfm_ctx* ctx) {
    CUDA_TRY(cudaSetDevice(ctx->device));
    return ESFM_OK;
}

template <typename T>
static int grow(T** ptr, size_t* cap_elems, size_t need_elems) {
    if (*cap_elems >= need_elems && *ptr) return ESFM_OK;
    if (*ptr) CUDA_TRY(cudaFree(*ptr));
    *ptr = nullptr;
    *cap_elems = 0;
    void* p = nullptr;
    cudaError_t e = cudaMalloc(&p, std::max<size_t>(need_elems, 1) * sizeof(T));
    if (e != cudaSuccess) { cudaGetLastError(); return fail(ESFM_ERR_NOMEM, "cudaMalloc(%zu bytes) failed: %s", need_elems * sizeof(T), cudaGetErrorString(e)); }
    *ptr = (T*)p;
    *cap_elems = need_elems;
    return ESFM_OK;
}

template <typename T>
static int grow_pinned(T** ptr, size_t* cap_elems, size_t need_elems) {
    if (*cap_elems >= need_elems && *ptr) return ESFM_OK;
    if (*ptr) CUDA_TRY(cudaFreeHost(*ptr));
    *ptr = nullptr;
    *cap_elems = 0;
    const size_t want = std::max<size_t>(need_elems + need_elems / 4, 4096);
    void* p = nullptr;
    cudaError_t e = cudaMallocHost(&p, want * sizeof(T));
    if (e != cudaSuccess) { cudaGetLastError(); return fail(ESFM_ERR_NOMEM, "cudaMallocHost(%zu bytes) failed: %s", want * sizeof(T), cudaGetErrorString(e)); }
    *ptr = (T*)p;
    *cap_elems = want;
    return ESFM_OK;
}

// stream-ordered allocation from the context's private pool
static cudaError_t pool_malloc(esfm_ctx* ctx, void** p, size_t bytes) {
    return cudaMallocFromPoolAsync(p, std::max<size_t>(bytes, 16), ctx->mempool, ctx->stream);
}

int esfm::reserve_stream_slots(esfm_ctx* ctx) {
    if (ctx->h_slot[0]) return ESFM_OK;
    CUDA_TRY(cudaSetDevice(ctx->device));
    for (int k = 0; k < esfm_ctx::kSlots; ++k) {
        cudaError_t e = cudaMallocHost((void**)&ctx->h_slot[k], esfm_ctx::kSlotMatches * sizeof(esfm_dmatch_t));
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ctx->ev_slot[k], cudaEventDisableTiming);
        if (e != cudaSuccess) { cudaGetLastError(); return fail(ESFM_ERR_NOMEM, "pinned stream slot allocation failed: %s", cudaGetErrorString(e)); }
    }
    return ESFM_OK;
}

// `n` matches from the device arena `src` to pageable host memory `dst`, through the pinned slots: the device->host copy of the
// next pieces runs (copy stream) while the helper threads move the current piece out of its slot.
static int stream_down(esfm_ctx* ctx, const esfm_dmatch_t* src, esfm_dmatch_t* dst, size_t n) {
    if (int rc = reserve_stream_slots(ctx)) return rc;
    const size_t P = esfm_ctx::kSlotMatches;
    const size_t pieces = (n + P - 1) / P;
    size_t issued = 0, done = 0;
    while (done < pieces) {
        while (issued < pieces && issued - done < (size_t)esfm_ctx::kSlots) {
            const size_t cnt = std::min(P, n - issued * P);
            const int sl = (int)(issued % esfm_ctx::kSlots);
            CUDA_TRY(cudaMemcpyAsync(ctx->h_slot[sl], src + issued * P, cnt * sizeof(esfm_dmatch_t), cudaMemcpyDeviceToHost, ctx->copy_stream));
            CUDA_TRY(cudaEventRecord(ctx->ev_slot[sl], ctx->copy_stream));
            ++issued;
        }
        const size_t cnt = std::min(P, n - done * P);
        const int sl = (int)(done % esfm_ctx::kSlots);
        CUDA_TRY(cudaEventSynchronize(ctx->ev_slot[sl]));
        ctx->copier->copy(dst + done * P, ctx->h_slot[sl], cnt * sizeof(esfm_dmatch_t));
        ++done;
    }
    ctx->stats.d2h_bytes += n * sizeof(esfm_dmatch_t);
    return ESFM_OK;
}

// ------------------------------------------------------------------------------------------------
// context
// ------------------------------------------------------------------------------------------------
extern "C" int esfm_abi_version(void) { return ESFM_ABI_VERSION; }
extern "C" const char* esfm_last_error(void) { return g_last_error.c_str(); }

extern "C" int esfm_init(int device, void* cuda_stream, esfm_ctx_t** out) {
    if (!out) return fail(ESFM_ERR_INVALID, "esfm_init: ctx is NULL");
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0)
        return fail(ESFM_ERR_CUDA, "esfm_init: no CUDA device (%s); this library has no CPU fallback",
                    e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
    if (device < 0 || device >= n) return fail(ESFM_ERR_INVALID, "esfm_init: device %d out of range [0,%d)", device, n);
    CUDA_TRY(cudaSetDevice(device));
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10)
        return fail(ESFM_ERR_CUDA, "esfm_init: device %d is sm_%d%d; this library is built for sm_100a (B200) only", device, prop.major, prop.minor);
    esfm_ctx* ctx = new (std::nothrow) esfm_ctx();
    if (!ctx) return fail(ESFM_ERR_NOMEM, "esfm_init: out of host memory");
    ctx->device = device;
    ctx->sm_count = prop.multiProcessorCount;
    if (const char* z = getenv("ESFM_ORB_Z")) ctx->orb_z = atoi(z) != 0;
    if (const char* z = getenv("ESFM_TC16_EXACT")) ctx->tc16_exact = atoi(z) != 0;
    if (const char* eng = getenv("ESFM_HAMMING_ENGINE")) {
        if (!strcmp(eng, "tc") || !strcmp(eng, "tensor")) ctx->hamming_engine = ESFM_HAMMING_ENGINE_TC;
        else if (!strcmp(eng, "tc16")) ctx->hamming_engine = ESFM_HAMMING_ENGINE_TC16;
        else if (!strcmp(eng, "popc")) ctx->hamming_engine = ESFM_HAMMING_ENGINE_POPC;
        else { delete ctx; return fail(ESFM_ERR_INVALID, "ESFM_HAMMING_ENGINE=%s: expected 'popc', 'tc' or 'tc16'", eng); }
    }
    if (const char* eng = getenv("ESFM_L2_ENGINE")) {
        if (!strcmp(eng, "tc") || !strcmp(eng, "tensor")) ctx->l2_engine = ESFM_L2_ENGINE_TC;
        else if (!strcmp(eng, "tc16")) ctx->l2_engine = ESFM_L2_ENGINE_TC16;
        else if (!strcmp(eng, "ffma")) ctx->l2_engine = ESFM_L2_ENGINE_FFMA;
        else { delete ctx; return fail(ESFM_ERR_INVALID, "ESFM_L2_ENGINE=%s: expected 'ffma', 'tc' or 'tc16'", eng); }
    }
    auto bail = [&](int code, const char* what, cudaError_t err) {
        const int rc = fail(code, "esfm_init: %s failed: %s", what, cudaGetErrorString(err));
        esfm_destroy(ctx);
        return rc;
    };
    if (cuda_stream) {
        ctx->stream = (cudaStream_t)cuda_stream;
    } else {
        e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking);
        if (e != cudaSuccess) return bail(ESFM_ERR_CUDA, "cudaStreamCreate", e);
        ctx->own_stream = true;
    }
    e = cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) return bail(ESFM_ERR_CUDA, "cudaStreamCreate", e);
    for (ChunkBuf& cb : ctx->buf) {
        for (cudaEvent_t* ev : {&cb.ev_t0, &cb.ev_t1, &cb.ev_t2, &cb.ev_v0, &cb.ev_v1}) {
            e = cudaEventCreate(ev);
            if (e != cudaSuccess) return bail(ESFM_ERR_CUDA, "cudaEventCreate", e);
        }
        for (cudaEvent_t* ev : {&cb.ev_meta, &cb.ev_copied}) {
            e = cudaEventCreateWithFlags(ev, cudaEventDisableTiming);
            if (e != cudaSuccess) return bail(ESFM_ERR_CUDA, "cudaEventCreate", e);
        }
        e = cudaMalloc((void**)&cb.d_cursor, 4 * sizeof(unsigned long long));
        if (e != cudaSuccess) return bail(ESFM_ERR_NOMEM, "cudaMalloc", e);
    }
    {   // banks come and go (one per all-pairs call in the per-call API): they are allocated stream-ordered from a memory pool
        // that keeps freed blocks cached, so steady state never pays cudaMalloc / cudaFree.  The pool is PRIVATE to the context
        // (the device's default pool is shared with everything else in the process, e.g. torch) and is destroyed with it.
        cudaMemPoolProps props{};
        props.allocType = cudaMemAllocationTypePinned;
        props.handleTypes = cudaMemHandleTypeNone;
        props.location.type = cudaMemLocationTypeDevice;
        props.location.id = device;
        e = cudaMemPoolCreate(&ctx->mempool, &props);
        if (e != cudaSuccess) return bail(ESFM_ERR_CUDA, "cudaMemPoolCreate", e);
        unsigned long long keep = ~0ull;
        cudaMemPoolSetAttribute(ctx->mempool, cudaMemPoolAttrReleaseThreshold, &keep);
    }
    int helpers = 3;
    if (const char* h = getenv("ESFM_COPY_THREADS")) helpers = std::max(0, std::min(15, atoi(h) - 1));
    ctx->copier = new (std::nothrow) CopyPool(helpers);
    if (!ctx->copier) { esfm_destroy(ctx); return fail(ESFM_ERR_NOMEM, "esfm_init: out of host memory"); }
    *out = ctx;
    return ESFM_OK;
}

extern "C" int esfm_destroy(esfm_ctx_t* ctx) {
    if (!ctx) return ESFM_OK;
    cudaSetDevice(ctx->device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    if (ctx->copy_stream) cudaStreamSynchronize(ctx->copy_stream);
    orb_state_destroy(ctx);
    for (esfm_bank*& pb : ctx->pair_bank) {
        if (pb) esfm_bank_destroy(pb);
        pb = nullptr;
    }
    cudaFree(ctx->keys);
    cudaFree(ctx->col_thr);
    cudaFree(ctx->gather_cnt);
    for (ChunkBuf& cb : ctx->buf) {
        cudaFree(cb.d_pairs); cudaFree(cb.d_pair_off); cudaFree(cb.d_pair_cnt); cudaFree(cb.d_cursor); cudaFree(cb.arena);
        if (cb.h_pairs) cudaFreeHost(cb.h_pairs);
        if (cb.h_meta) cudaFreeHost(cb.h_meta);
        for (cudaEvent_t ev : {cb.ev_t0, cb.ev_t1, cb.ev_t2, cb.ev_v0, cb.ev_v1, cb.ev_meta, cb.ev_copied})
            if (ev) cudaEventDestroy(ev);
    }
    for (auto& b : ctx->pool) cudaFreeHost(b.ptr);
    for (int k = 0; k < esfm_ctx::kSlots; ++k) {
        if (ctx->h_slot[k]) cudaFreeHost(ctx->h_slot[k]);
        if (ctx->ev_slot[k]) cudaEventDestroy(ctx->ev_slot[k]);
    }
    free(ctx->h_scratch);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);     // (the stream-ordered frees of the pair banks)
    if (ctx->mempool) cudaMemPoolDestroy(ctx->mempool);
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx->copier;
    delete ctx;
    return ESFM_OK;
}

extern "C" int esfm_synchronize(esfm_ctx_t* ctx) {
    if (!ctx) return fail(ESFM_ERR_INVALID, "ctx is NULL");
    if (int rc = set_device(ctx)) return rc;
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->copy_stream));
    return ESFM_OK;
}

extern "C" int esfm_get_stats(esfm_ctx_t* ctx, esfm_stats_t* out) {
    if (!ctx || !out) return fail(ESFM_ERR_INVALID, "esfm_get_stats: NULL argument");
    *out = ctx->stats;
    return ESFM_OK;
}

extern "C" int esfm_set_profiling(esfm_ctx_t* ctx, int enabled) {
    if (!ctx) return fail(ESFM_ERR_INVALID, "ctx is NULL");
    ctx->profiling = enabled != 0;
    return ESFM_OK;
}

extern "C" int esfm_set_l2_engine(esfm_ctx_t* ctx, int engine) {
    if (!ctx) return fail(ESFM_ERR_INVALID, "ctx is NULL");
    if (engine != ESFM_L2_ENGINE_FFMA && engine != ESFM_L2_ENGINE_TC && engine != ESFM_L2_ENGINE_TC16) return fail(ESFM_ERR_INVALID, "unknown L2 engine %d", engine);
    ctx->l2_engine = engine;
    return ESFM_OK;
}

extern "C" int esfm_set_hamming_engine(esfm_ctx_t* ctx, int engine) {
    if (!ctx) return fail(ESFM_ERR_INVALID, "ctx is NULL");
    if (engine != ESFM_HAMMING_ENGINE_POPC && engine != ESFM_HAMMING_ENGINE_TC && engine != ESFM_HAMMING_ENGINE_TC16) return fail(ESFM_ERR_INVALID, "unknown Hamming engine %d", engine);
    ctx->hamming_engine = engine;
    return ESFM_OK;
}

extern "C" int esfm_get_hamming_engine(esfm_ctx_t* ctx, int* engine) {
    if (!ctx || !engine) return fail(ESFM_ERR_INVALID, "esfm_get_hamming_engine: NULL argument");
    *engine = ctx->hamming_engine;
    return ESFM_OK;
}

extern "C" int esfm_get_l2_engine(esfm_ctx_t* ctx, int* engine) {
    if (!ctx || !engine) return fail(ESFM_ERR_INVALID, "esfm_get_l2_engine: NULL argument");
    *engine = ctx->l2_engine;
    return ESFM_OK;
}

extern "C" int esfm_device_sm_count(esfm_ctx_t* ctx, int* sms) {
    if (!ctx || !sms) return fail(ESFM_ERR_INVALID, "esfm_device_sm_count: NULL argument");
    *sms = ctx->sm_count;
    return ESFM_OK;
}

// ------------------------------------------------------------------------------------------------
// bank
// ------------------------------------------------------------------------------------------------
extern "C" int esfm_bank_create(esfm_ctx_t* ctx, esfm_kind kind, int n_frames, esfm_bank_t** out) {
    if (!ctx || !out) return fail(ESFM_ERR_INVALID, "esfm_bank_create: NULL argument");
    *out = nullptr;
    if (kind != ESFM_KIND_F32X64 && kind != ESFM_KIND_B256) return fail(ESFM_ERR_INVALID, "esfm_bank_create: unknown kind %d", (int)kind);
    if (n_frames < 0) return fail(ESFM_ERR_INVALID, "esfm_bank_create: n_frames < 0");
    esfm_bank* b = new (std::nothrow) esfm_bank();
    if (!b) return fail(ESFM_ERR_NOMEM, "out of host memory");
    b->ctx = ctx;
    b->kind = kind;
    b->n_frames = n_frames;
    b->rows.assign(n_frames, -1);
    b->host_off.assign(n_frames, (size_t)-1);
    b->host_ext.assign(n_frames, nullptr);
    *out = b;
    return ESFM_OK;
}

static int check_frame_limits(esfm_bank* b, int rows) {
    const int lim = b->kind == ESFM_KIND_F32X64 ? sweep_l2_max_rows() : sweep_hamming_max_rows();
    if (rows > lim) return fail(ESFM_ERR_CAPACITY, "frame has %d rows; this build supports at most %d per frame for kind %d", rows, lim, b->kind);
    return ESFM_OK;
}

static int check_set_frame_args(esfm_bank* b, const char* who, int frame_id, const void* data, int rows, int cols) {
    if (b->committed || b->device_allocated) return fail(ESFM_ERR_STATE, "%s: bank already committed", who);
    if (frame_id < 0 || frame_id >= b->n_frames) return fail(ESFM_ERR_INVALID, "frame_id %d out of range [0,%d)", frame_id, b->n_frames);
    if (rows < 0) return fail(ESFM_ERR_INVALID, "rows < 0");
    const int want_cols = b->kind == ESFM_KIND_F32X64 ? kDim : 32;
    if (rows > 0 && cols != want_cols)
        return fail(ESFM_ERR_INVALID, "kind %d needs %d columns per descriptor, got %d", b->kind, want_cols, cols);
    if (rows > 0 && !data) return fail(ESFM_ERR_INVALID, "data is NULL with rows > 0");
    return check_frame_limits(b, rows);
}

// Grow the staging pair (pinned host buffer + its device mirror) to hold `need` more bytes.
static int staging_reserve(esfm_bank* b, size_t need) {
    if (b->up_used + need <= b->up_cap) return ESFM_OK;
    esfm_ctx* ctx = b->ctx;
    // first growth after the first frame: assume the other frames are about as large (the reference's frames all come from
    // one extractor setting, feature_matching.cpp:16-22,45-52), so a whole bank normally needs ONE staging allocation
    size_t want = std::max((b->up_used + need) * 2, (size_t)8 << 20);
    if (b->up_cap == 0 && b->n_frames > 1) want = std::max(want, (size_t)((double)need * b->n_frames * 1.05) + ((size_t)1 << 20));
    size_t cap = 0;
    uint8_t* nh = (uint8_t*)pool_acquire(ctx, want, &cap);
    if (!nh) return fail(ESFM_ERR_NOMEM, "pinned staging allocation of %zu bytes failed", want);
    uint8_t* nd = nullptr;
    // + one tile of slack so that the mirror can become the bank itself (tile-granular reads past the last frame)
    cudaError_t e = pool_malloc(ctx, (void**)&nd, cap + (size_t)kHamTile * b->row_bytes());
    if (e != cudaSuccess) { cudaGetLastError(); pool_release(ctx, nh); return fail(ESFM_ERR_NOMEM, "cudaMallocAsync(%zu) for the upload mirror failed: %s", cap, cudaGetErrorString(e)); }
    if (b->up_used) {
        // frames already staged: in-flight host->device copies still read the old pinned buffer
        CUDA_TRY(cudaStreamSynchronize(ctx->stream));
        memcpy(nh, b->h_up, b->up_used);
        CUDA_TRY(cudaMemcpyAsync(nd, b->d_up, b->up_used, cudaMemcpyDeviceToDevice, ctx->stream));
    }
    if (b->d_up) cudaFreeAsync(b->d_up, ctx->stream);
    pool_release(ctx, b->h_up);
    b->h_up = nh;
    b->d_up = nd;
    b->up_cap = cap;
    return ESFM_OK;
}

extern "C" int esfm_bank_set_frame(esfm_bank_t* b, int frame_id, const void* data, int rows, int cols, size_t step_bytes) {
    if (!b) return fail(ESFM_ERR_INVALID, "bank is NULL");
    if (int rc = check_set_frame_args(b, "esfm_bank_set_frame", frame_id, data, rows, cols)) return rc;
    const size_t rb = b->row_bytes();
    if (rows > 0 && step_bytes < rb) return fail(ESFM_ERR_INVALID, "step_bytes %zu smaller than a row (%zu)", step_bytes, rb);
    esfm_ctx* ctx = b->ctx;
    if (int rc = set_device(ctx)) return rc;
    const size_t need = (size_t)rows * rb;
    if (int rc = staging_reserve(b, need)) return rc;
    uint8_t* dst = b->h_up + b->up_used;
    if (step_bytes == rb) {
        ctx->copier->copy(dst, data, need);
    } else {
        for (int r = 0; r < rows; ++r) memcpy(dst + (size_t)r * rb, (const uint8_t*)data + (size_t)r * step_bytes, rb);
    }
    // the caller's memory is pageable (cv::Mat) and need not outlive the call: the frame now sits in pinned staging, and its
    // host->device copy starts at once -- it runs while the caller prepares / this function stages the next frame
    if (need) {
        CUDA_TRY(cudaMemcpyAsync(b->d_up + b->up_used, dst, need, cudaMemcpyHostToDevice, ctx->stream));
        ctx->stats.h2d_bytes += need;
    }
    b->host_off[frame_id] = b->up_used;
    b->host_ext[frame_id] = nullptr;
    b->up_used += need;
    b->rows[frame_id] = rows;
    return ESFM_OK;
}

// ORB extraction straight into the bank (orb.cu): the descriptors are produced on the device and land in the upload mirror at the place
// esfm_bank_set_frame would have copied them to; the pinned half of the staging pair stays unwritten for this frame (esfm_bank_commit reads
// staged frames from the mirror only).
extern "C" int esfm_bank_set_frame_from_image(esfm_bank_t* b, int frame_id, const unsigned char* image, int rows, int cols, int channels,
                                              size_t row_stride, int max_features, esfm_keypoint_t* keypoints, unsigned char* descriptors_host,
                                              int capacity, int* n_out) {
    if (!b) return fail(ESFM_ERR_INVALID, "bank is NULL");
    if (b->kind != ESFM_KIND_B256) return fail(ESFM_ERR_INVALID, "esfm_bank_set_frame_from_image needs a B256 bank");
    if (b->committed || b->device_allocated) return fail(ESFM_ERR_STATE, "esfm_bank_set_frame_from_image: bank already committed");
    if (frame_id < 0 || frame_id >= b->n_frames) return fail(ESFM_ERR_INVALID, "frame_id %d out of range [0,%d)", frame_id, b->n_frames);
    esfm_ctx* ctx = b->ctx;
    size_t at = 0;
    const OrbSink sink = [&](int n, uint8_t** d_dst) -> int {
        if (int rc = check_frame_limits(b, n)) return rc;
        if (int rc = staging_reserve(b, (size_t)n * 32)) return rc;
        at = b->up_used;
        *d_dst = b->d_up + at;
        return ESFM_OK;
    };
    int n = 0;
    if (int rc = orb_extract_impl(ctx, image, rows, cols, channels, row_stride, max_features, keypoints, descriptors_host, capacity, &n, sink)) {
        if (n_out) *n_out = n;
        return rc;
    }
    if (n_out) *n_out = n;
    b->host_off[frame_id] = at;
    b->host_ext[frame_id] = nullptr;
    b->up_used = at + (size_t)n * 32;
    b->rows[frame_id] = n;
    return ESFM_OK;
}

extern "C" int esfm_bank_set_frame_pinned(esfm_bank_t* b, int frame_id, const void* data, int rows, int cols, size_t step_bytes) {
    if (!b) return fail(ESFM_ERR_INVALID, "bank is NULL");
    if (int rc = check_set_frame_args(b, "esfm_bank_set_frame_pinned", frame_id, data, rows, cols)) return rc;
    if (rows > 0 && step_bytes != b->row_bytes())
        return fail(ESFM_ERR_INVALID, "esfm_bank_set_frame_pinned needs densely packed rows (step_bytes %zu != %zu)", step_bytes, b->row_bytes());
    if (rows > 0) {
        if (int rc = set_device(b->ctx)) return rc;
        cudaPointerAttributes at{};
        const cudaError_t e = cudaPointerGetAttributes(&at, data);
        if (e != cudaSuccess || at.type != cudaMemoryTypeHost) {
            cudaGetLastError();
            return fail(ESFM_ERR_INVALID, "esfm_bank_set_frame_pinned: frame %d is not in page-locked host memory", frame_id);
        }
    }
    b->host_off[frame_id] = (size_t)-1;
    b->host_ext[frame_id] = rows > 0 ? data : nullptr;
    b->rows[frame_id] = rows;
    return ESFM_OK;
}

extern "C" int esfm_bank_set_frame_rows(esfm_bank_t* b, int frame_id, int rows) {
    if (!b) return fail(ESFM_ERR_INVALID, "bank is NULL");
    if (b->committed || b->device_allocated) return fail(ESFM_ERR_STATE, "bank already committed");
    if (frame_id < 0 || frame_id >= b->n_frames) return fail(ESFM_ERR_INVALID, "frame_id %d out of range", frame_id);
    if (rows < 0) return fail(ESFM_ERR_INVALID, "rows < 0");
    if (int rc = check_frame_limits(b, rows)) return rc;
    b->rows[frame_id] = rows;
    b->host_off[frame_id] = (size_t)-1;
    b->host_ext[frame_id] = nullptr;
    return ESFM_OK;
}

// Row / tile offsets of the declared frames, the raw row-major device buffer (the upload mirror itself when it already IS
// that buffer) and the three offset tables on the device.
static int bank_alloc_layout(esfm_bank* b, bool adopt_mirror) {
    esfm_ctx* ctx = b->ctx;
    if (int rc = set_device(ctx)) return rc;
    for (int f = 0; f < b->n_frames; ++f)
        if (b->rows[f] < 0) return fail(ESFM_ERR_STATE, "frame %d was never set", f);
    b->row_off.assign(b->n_frames + 1, 0);
    b->tile_off.assign(b->n_frames + 1, 0);
    b->max_rows = 0;
    for (int f = 0; f < b->n_frames; ++f) {
        b->row_off[f + 1] = b->row_off[f] + b->rows[f];
        b->tile_off[f + 1] = b->tile_off[f] + (b->rows[f] + kTile - 1) / kTile;
        b->max_rows = std::max(b->max_rows, b->rows[f]);
        if (b->row_off[f + 1] < b->row_off[f]) return fail(ESFM_ERR_CAPACITY, "bank exceeds 2^31 rows");
    }
    const size_t total_rows = (size_t)b->row_off[b->n_frames];
    // one extra tile of slack so tile-granular reads past the last frame stay inside the allocation
    b->rows_bytes = (total_rows + kHamTile) * b->row_bytes();
    if (adopt_mirror && b->d_up && b->up_cap + (size_t)kHamTile * b->row_bytes() >= b->rows_bytes) {
        if (b->d_rows && b->d_rows != b->d_up) cudaFreeAsync(b->d_rows, ctx->stream);
        b->d_rows = b->d_up;
        b->rows_cap = b->up_cap + (size_t)kHamTile * b->row_bytes();
    } else if (!b->d_rows || b->d_rows == b->d_up || b->rows_cap < b->rows_bytes) {
        if (b->d_rows && b->d_rows != b->d_up) cudaFreeAsync(b->d_rows, ctx->stream);
        b->d_rows = nullptr;
        cudaError_t e = pool_malloc(ctx, &b->d_rows, b->rows_bytes);
        if (e != cudaSuccess) { cudaGetLastError(); return fail(ESFM_ERR_NOMEM, "cudaMallocAsync(%zu) for the descriptor bank failed: %s", b->rows_bytes, cudaGetErrorString(e)); }
        b->rows_cap = b->rows_bytes;
    }
    // only the slack past the last frame needs defined contents
    CUDA_TRY(cudaMemsetAsync((uint8_t*)b->d_rows + total_rows * b->row_bytes(), 0, (size_t)kHamTile * b->row_bytes(), ctx->stream));
    const size_t ne = (size_t)(b->n_frames + 1);
    if (!b->d_tables) {
        cudaError_t e = pool_malloc(ctx, (void**)&b->d_tables, 4 * ne * sizeof(int));   // + per frame the largest |x| (bank_check_range)
        if (e != cudaSuccess) { cudaGetLastError(); return fail(ESFM_ERR_NOMEM, "cudaMallocAsync for the frame tables failed: %s", cudaGetErrorString(e)); }
        b->d_frame_rows = b->d_tables;
        b->d_row_off = b->d_tables + ne;
        b->d_tile_off = b->d_tables + 2 * ne;
    }
    // one small upload: rows | row_off | tile_off (pageable source: the copy has left the host buffer when the call returns)
    std::vector<int> tab(3 * ne, 0);
    std::copy(b->rows.begin(), b->rows.end(), tab.begin());
    std::copy(b->row_off.begin(), b->row_off.end(), tab.begin() + ne);
    std::copy(b->tile_off.begin(), b->tile_off.end(), tab.begin() + 2 * ne);
    CUDA_TRY(cudaMemcpyAsync(b->d_tables, tab.data(), tab.size() * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    ctx->stats.h2d_bytes += tab.size() * sizeof(int);
    b->device_allocated = true;
    b->kmajor_built = b->tc_built = false;
    return ESFM_OK;
}

extern "C" int esfm_bank_alloc_device(esfm_bank_t* b) {
    if (!b) return fail(ESFM_ERR_INVALID, "bank is NULL");
    if (b->device_allocated) return fail(ESFM_ERR_STATE, "bank already allocated");
    return bank_alloc_layout(b, false);
}

// Give the staging buffers back (the host side to the context's pool, the device mirror unless it became the bank).
static void bank_release_staging(esfm_bank* b) {
    esfm_ctx* ctx = b->ctx;
    pool_release(ctx, b->h_up);
    b->h_up = nullptr;
    if (b->d_up && b->d_up != b->d_rows) cudaFreeAsync(b->d_up, ctx->stream);
    b->d_up = nullptr;
    b->up_cap = b->up_used = 0;
}

// F32X64: the input range of the committed rows (frame_absmax_kernel; set_frame_pinned and commit_device data never pass through host
// staging, so it is measured on the device), which plan_sweep routes on.  Non-finite components, for which L2 matching has no defined answer,
// and magnitudes beyond every engine's range are refused.
static int bank_check_range(esfm_bank* b) {
    if (b->kind != ESFM_KIND_F32X64) return ESFM_OK;
    esfm_ctx* ctx = b->ctx;
    const size_t ne = (size_t)(b->n_frames + 1);
    unsigned* d_absmax = reinterpret_cast<unsigned*>(b->d_tables + 3 * ne);
    CUDA_TRY(launch_frame_absmax((const float*)b->d_rows, b->d_frame_rows, b->d_row_off, b->d_tile_off, b->n_frames, b->tile_off[b->n_frames],
                                 d_absmax, ctx->stream));
    std::vector<unsigned> bits(b->n_frames);
    CUDA_TRY(cudaMemcpyAsync(bits.data(), d_absmax, bits.size() * sizeof(unsigned), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    b->abs_max = 0.f;
    b->frame_abs_min = INFINITY;
    for (int f = 0; f < b->n_frames; ++f) {
        if (b->rows[f] == 0) continue;
        if (bits[f] >= 0x7f800000u) return fail(ESFM_ERR_INVALID, "frame %d has a non-finite (inf or NaN) component: L2 matching has no defined answer for it", f);
        float m;
        memcpy(&m, &bits[f], sizeof m);
        if (m > kFfmaMaxAbs)
            return fail(ESFM_ERR_INVALID, "frame %d has a component of magnitude %g; L2 matching supports |x| <= 2^59 (%g), where squared distances "
                                          "stay finite in fp32", f, m, kFfmaMaxAbs);
        b->abs_max = std::max(b->abs_max, m);
        b->frame_abs_min = std::min(b->frame_abs_min, m);
    }
    return ESFM_OK;
}

extern "C" int esfm_bank_commit(esfm_bank_t* b) {
    if (!b) return fail(ESFM_ERR_INVALID, "bank is NULL");
    if (b->committed) return fail(ESFM_ERR_STATE, "bank already committed");
    for (int f = 0; f < b->n_frames; ++f)     // (also after esfm_bank_alloc_device: there is no host data to copy then)
        if (b->rows[f] > 0 && b->host_off[f] == (size_t)-1 && !b->host_ext[f])
            return fail(ESFM_ERR_STATE, "frame %d has rows declared but no host data; use esfm_bank_alloc_device + esfm_bank_commit_device", f);
    if (b->device_allocated) return fail(ESFM_ERR_STATE, "bank storage was allocated with esfm_bank_alloc_device: finish with esfm_bank_commit_device");
    esfm_ctx* ctx = b->ctx;
    if (int rc = set_device(ctx)) return rc;
    const size_t rb = b->row_bytes();
    // frames staged in order (the normal case) have ALREADY been copied into the mirror exactly where the bank wants them
    bool in_order = true;
    size_t expect = 0;
    for (int f = 0; f < b->n_frames && in_order; ++f) {
        if (b->rows[f] < 0) return fail(ESFM_ERR_STATE, "frame %d was never set", f);
        if (b->rows[f] > 0 && (b->host_ext[f] || b->host_off[f] != expect)) in_order = false;
        expect += (size_t)b->rows[f] * rb;
    }
    in_order = in_order && expect == b->up_used;
    if (int rc = bank_alloc_layout(b, in_order)) return rc;
    if (!in_order) {      // frames were set out of order, re-set, or come from caller-owned pinned memory: one copy per frame
        for (int f = 0; f < b->n_frames; ++f) {
            if (b->rows[f] <= 0) continue;
            uint8_t* dst = (uint8_t*)b->d_rows + (size_t)b->row_off[f] * rb;
            const size_t bytes = (size_t)b->rows[f] * rb;
            if (b->host_ext[f]) {
                CUDA_TRY(cudaMemcpyAsync(dst, b->host_ext[f], bytes, cudaMemcpyHostToDevice, ctx->stream));
                ctx->stats.h2d_bytes += bytes;
            } else {
                CUDA_TRY(cudaMemcpyAsync(dst, b->d_up + b->host_off[f], bytes, cudaMemcpyDeviceToDevice, ctx->stream));
            }
        }
    }
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));   // uploads done: pinned sources (ours and the caller's) are free again
    bank_release_staging(b);
    if (int rc = bank_check_range(b)) return rc;
    b->committed = true;
    return ESFM_OK;
}

extern "C" int esfm_bank_device_rows(esfm_bank_t* b, void** dev_ptr, size_t* bytes) {
    if (!b || !dev_ptr || !bytes) return fail(ESFM_ERR_INVALID, "esfm_bank_device_rows: NULL argument");
    if (!b->device_allocated) return fail(ESFM_ERR_STATE, "bank has no device storage yet");
    *dev_ptr = b->d_rows;
    *bytes = (size_t)b->row_off[b->n_frames] * b->row_bytes();
    return ESFM_OK;
}

extern "C" int esfm_bank_commit_device(esfm_bank_t* b) {
    if (!b) return fail(ESFM_ERR_INVALID, "bank is NULL");
    if (!b->device_allocated) return fail(ESFM_ERR_STATE, "call esfm_bank_alloc_device first");
    if (int rc = set_device(b->ctx)) return rc;
    CUDA_TRY(cudaStreamSynchronize(b->ctx->stream));
    b->kmajor_built = b->tc_built = false;          // the raw rows may have been rewritten
    if (int rc = bank_check_range(b)) return rc;
    b->committed = true;
    return ESFM_OK;
}

extern "C" int esfm_bank_n_frames(esfm_bank_t* b, int* n) {
    if (!b || !n) return fail(ESFM_ERR_INVALID, "NULL argument");
    *n = b->n_frames;
    return ESFM_OK;
}

extern "C" int esfm_bank_frame_rows(esfm_bank_t* b, int frame_id, int* rows) {
    if (!b || !rows) return fail(ESFM_ERR_INVALID, "NULL argument");
    if (frame_id < 0 || frame_id >= b->n_frames) return fail(ESFM_ERR_INVALID, "frame_id %d out of range", frame_id);
    *rows = b->rows[frame_id];
    return ESFM_OK;
}

extern "C" int esfm_bank_device_bytes(esfm_bank_t* b, size_t* bytes) {
    if (!b || !bytes) return fail(ESFM_ERR_INVALID, "NULL argument");
    *bytes = b->device_allocated ? b->rows_bytes + (b->kmajor_built ? b->kmajor_bytes : 0) + (b->tc_built ? b->tc_bytes : 0) : 0;
    return ESFM_OK;
}

extern "C" int esfm_bank_destroy(esfm_bank_t* b) {
    if (!b) return ESFM_OK;
    if (b->ctx) {
        cudaSetDevice(b->ctx->device);
        cudaStream_t s = b->ctx->stream;   // stream-ordered frees: queued behind any work still using the bank
        if (b->d_up && b->d_up != b->d_rows) cudaFreeAsync(b->d_up, s);
        if (b->d_rows) cudaFreeAsync(b->d_rows, s);
        if (b->d_kmajor) cudaFreeAsync(b->d_kmajor, s);
        if (b->d_tc) cudaFreeAsync(b->d_tc, s);
        if (b->d_tables) cudaFreeAsync(b->d_tables, s);
        if (b->h_up) {
            cudaStreamSynchronize(s);      // staged frames may still be on their way to the mirror
            pool_release(b->ctx, b->h_up);
        }
    }
    delete b;
    return ESFM_OK;
}

// Back to "created": every frame unset, device buffers kept for the next fill (esfm_match_descriptors reuses one two-frame
// bank per kind instead of allocating and freeing five device buffers per image pair).
static void bank_reset(esfm_bank* b) {
    esfm_ctx* ctx = b->ctx;
    std::fill(b->rows.begin(), b->rows.end(), -1);
    std::fill(b->host_off.begin(), b->host_off.end(), (size_t)-1);
    std::fill(b->host_ext.begin(), b->host_ext.end(), nullptr);
    if (b->d_rows && !b->d_up) {            // the device buffer of the last fill becomes the upload mirror of the next one
        const size_t slack = (size_t)kHamTile * b->row_bytes();
        size_t cap = 0;
        uint8_t* nh = b->rows_cap > slack ? (uint8_t*)pool_acquire(ctx, b->rows_cap - slack, &cap) : nullptr;
        if (nh) {                           // (steady state: the pinned buffer the last commit gave back to the pool)
            b->h_up = nh;
            b->d_up = (uint8_t*)b->d_rows;
            b->up_cap = b->rows_cap - slack;
        } else {
            cudaFreeAsync(b->d_rows, ctx->stream);
        }
        b->d_rows = nullptr;
        b->rows_cap = 0;
    }
    b->up_used = 0;
    b->committed = b->device_allocated = false;
    b->kmajor_built = b->tc_built = false;
}

// ------------------------------------------------------------------------------------------------
// matching
// ------------------------------------------------------------------------------------------------
namespace {

struct ChunkPlan {
    int stride;        // keys per array
    int col_cap;       // smem threshold entries
    size_t chunk_pairs;
};

// The sweep kernels: sweep_l2.cu, sweep_hamming.cu, sweep_l2_tc.cu (rows and column minima in one sweep), sweep_win.cu (rows only, slice keys)
enum class SweepKind { Ffma, Popc, Tc, Win };

// How one chunk is swept: the kernel, what it needs from the bank and the scratch, and how finalize reads its keys
struct SweepPlan {
    SweepKind sweep;
    TcImage image;                              // operand image of the bank (Tc, Win)
    int thr_fill = -1;                          // byte the column thresholds start at; -1: the sweep reads none
    KeyFormat key_format = KeyFormat::Direct;
    bool fast;           // SURF Win: fast mode, then an exact fallback sweep of the rows its error bound cannot settle
    bool two_phase;      // Win cross-check: ratio test, then a verification sweep of the undecided train rows (finalize.cu)
};

// A SURF bank is swept by the context's engine when its components lie inside that engine's input range (esfm_internal.cuh), else by the
// next engine that covers them: tc16 -> tc -> ffma (esfm_bank_commit has refused banks outside ffma's range).
static int l2_engine_for(const esfm_bank* b, int engine) {
    if (engine == ESFM_L2_ENGINE_TC16 && !(b->abs_max <= kTc16MaxAbs && b->frame_abs_min >= kTc16MinFrameAbs)) engine = ESFM_L2_ENGINE_TC;
    if (engine == ESFM_L2_ENGINE_TC && !(b->abs_max <= kTcMaxAbs)) engine = ESFM_L2_ENGINE_FFMA;
    return engine;
}

// The tc16 sweeps (sweep_win.cu) are ROWS-ONLY.  Their cross-check runs in TWO PHASES: (1) the rows-only sweep + ratio test, survivors
// claim their train rows and histograms of every row's best / second-best value decide which survivors could still be beaten; (2) a
// second rows-only sweep with the roles swapped over just the undecided train rows (gathered into the query operand), whose answer --
// the nearest query row of each -- settles them.  Raw knn output (esfm_knn2_pair) needs column minima inside ONE sweep: a tc16 context
// runs it on the fp32-accumulator sweep of sweep_l2_tc.cu (the bank's operand image is rebuilt on the switch).
SweepPlan plan_sweep(const esfm_ctx* ctx, const esfm_bank* b, bool cross_check, bool knn) {
    const bool surf = b->kind == ESFM_KIND_F32X64;
    const int engine = surf ? l2_engine_for(b, ctx->l2_engine) : ctx->hamming_engine;
    SweepPlan s{};
    if (engine == (surf ? ESFM_L2_ENGINE_FFMA : ESFM_HAMMING_ENGINE_POPC)) {
        s.sweep = surf ? SweepKind::Ffma : SweepKind::Popc;
        if (surf) s.thr_fill = kThrInit & 0xff;      // (the POPC sweep keeps its column minima in shared memory)
    } else if (engine == (surf ? ESFM_L2_ENGINE_TC16 : ESFM_HAMMING_ENGINE_TC16) && !knn) {
        s.sweep = SweepKind::Win;                     // (col_thr only holds its gather lists)
        s.image = surf ? TcImage::H : TcImage::Fp8Pm1;
        s.key_format = KeyFormat::Slice;
        s.fast = surf && !ctx->tc16_exact;
        s.two_phase = cross_check;
    } else {
        s.sweep = SweepKind::Tc;
        if (surf) {
            s.image = TcImage::Tf32x3;
            s.thr_fill = kTcBoundBitsF32 & 0xff;
        } else if (ctx->orb_z && b->max_rows <= kTcZMaxRows) {     // the column index rides in the Z key: at most 2^15 rows per frame
            s.image = TcImage::Fp8Z;
            s.thr_fill = kTcBoundBitsZ & 0xff;
            s.key_format = KeyFormat::TcZ;
        } else {
            s.image = TcImage::Fp8Pm1;
            s.thr_fill = kTcBoundBitsB256 & 0xff;
            s.key_format = KeyFormat::TcPm1;
        }
    }
    return s;
}

ChunkPlan plan_chunks(const esfm_bank* b, int64_t n_pairs) {
    ChunkPlan pl;
    const int padded = ((b->max_rows + kTile - 1) / kTile) * kTile;
    pl.stride = std::max(padded, kTile);
    pl.col_cap = pl.stride;
    const size_t key_bytes_per_pair = (size_t)4 * pl.stride * sizeof(u64);
    const size_t arena_bytes_per_pair = (size_t)std::max(b->max_rows, 1) * sizeof(esfm_dmatch_t);
    const size_t budget_keys = (size_t)4 << 30, budget_arena = (size_t)2 << 30;
    size_t c = std::min(budget_keys / key_bytes_per_pair, budget_arena / arena_bytes_per_pair);
    // (Measured: splitting a batch that fits in one or two chunks into four equal ones to overlap more of the match download LOSES -- ORB e2e
    // 3.99e12 -> 3.38e12 comparisons/s: per-chunk launches, synchronisations and the pinned-slot streaming cost more than the exposed copy.)
    c = std::max<size_t>(1, std::min<size_t>(c, 65536));
    if (const char* e = getenv("ESFM_CHUNK_PAIRS")) c = std::max<size_t>(1, std::min<size_t>(c, (size_t)atoll(e)));   // tests: force several chunks
    pl.chunk_pairs = (size_t)std::min<int64_t>((int64_t)c, std::max<int64_t>(n_pairs, 1));
    return pl;
}

int ensure_scratch(esfm_ctx* ctx, const esfm_bank* b, const SweepPlan& sw, const ChunkPlan& pl, int n_bufs) {
    size_t key_elems = pl.chunk_pairs * 4 * (size_t)pl.stride;
    size_t cap = ctx->keys_bytes / sizeof(u64);
    if (int rc = grow(&ctx->keys, &cap, key_elems)) return rc;
    ctx->keys_bytes = cap * sizeof(u64);
    if (sw.sweep != SweepKind::Popc)
        if (int rc = grow(&ctx->col_thr, &ctx->col_thr_elems, pl.chunk_pairs * (size_t)pl.stride)) return rc;
    if (sw.sweep == SweepKind::Win)
        if (int rc = grow(&ctx->gather_cnt, &ctx->gather_cnt_elems, pl.chunk_pairs)) return rc;
    const size_t arena_need = pl.chunk_pairs * (size_t)std::max(b->max_rows, 1);
    for (int k = 0; k < n_bufs; ++k) {
        ChunkBuf& cb = ctx->buf[k];
        if (cb.copy_pending) {            // an earlier batch's copy may still read this arena
            CUDA_TRY(cudaEventSynchronize(cb.ev_copied));
            cb.copy_pending = false;
        }
        if (int rc = grow(&cb.arena, &cb.arena_cap, arena_need)) return rc;
        if (cb.pairs_cap < pl.chunk_pairs) {
            size_t c1 = cb.pairs_cap, c2 = cb.pairs_cap, c3 = cb.pairs_cap;
            if (int rc = grow(&cb.d_pairs, &c1, pl.chunk_pairs)) return rc;
            if (int rc = grow(&cb.d_pair_off, &c2, pl.chunk_pairs)) return rc;
            if (int rc = grow(&cb.d_pair_cnt, &c3, pl.chunk_pairs)) return rc;
            cb.pairs_cap = pl.chunk_pairs;
        }
        if (int rc = grow_pinned(&cb.h_pairs, &cb.h_pairs_cap, pl.chunk_pairs)) return rc;
        const size_t meta = pl.chunk_pairs * (sizeof(int32_t) + sizeof(unsigned long long)) + 4 * sizeof(unsigned long long);
        if (int rc = grow_pinned(&cb.h_meta, &cb.h_meta_bytes, meta)) return rc;
    }
    return ESFM_OK;
}

// Derived operand layouts, each built the first time an engine that reads it sweeps the bank.
// FFMA engine: k-major 128-row tiles + half squared norms.
int ensure_kmajor_layout(esfm_ctx* ctx, esfm_bank* b) {
    if (b->kmajor_built) return ESFM_OK;
    const int n_tiles = b->tile_off[b->n_frames];
    b->kmajor_bytes = ((size_t)n_tiles + 1) * kTileBytes;
    if (!b->d_kmajor || b->kmajor_cap < b->kmajor_bytes) {
        if (b->d_kmajor) cudaFreeAsync(b->d_kmajor, ctx->stream);
        b->d_kmajor = nullptr;
        cudaError_t e = pool_malloc(ctx, (void**)&b->d_kmajor, b->kmajor_bytes);
        if (e != cudaSuccess) { cudaGetLastError(); return fail(ESFM_ERR_NOMEM, "cudaMallocAsync(%zu) for the k-major bank failed: %s", b->kmajor_bytes, cudaGetErrorString(e)); }
        b->kmajor_cap = b->kmajor_bytes;
    }
    cudaError_t e = launch_pack_f32((const float*)b->d_rows, b->d_frame_rows, b->d_row_off, b->d_tile_off, b->n_frames, n_tiles, b->d_kmajor, ctx->stream);
    if (e != cudaSuccess) return fail(ESFM_ERR_CUDA, "pack_f32 kernel launch failed: %s", cudaGetErrorString(e));
    if (n_tiles > 0) ctx->stats.kernel_launches += 1;
    b->kmajor_built = true;
    return ESFM_OK;
}

// Tensor-core engines: the operand images of tc_layout.cuh (TcImage).
// The H images are followed by what win_fast_eps needs: float row_eps[total rows], frame_norm[n_frames].
float* tch_row_eps(const esfm_bank* b) { return reinterpret_cast<float*>(b->d_tc + ((size_t)b->tile_off[b->n_frames] + 1) * kTchTileBytes); }
float* tch_frame_norm(const esfm_bank* b) { return tch_row_eps(b) + b->row_off[b->n_frames]; }

int ensure_tc_layout(esfm_ctx* ctx, esfm_bank* b, TcImage img) {
    if (b->tc_built && b->tc_image == img) return ESFM_OK;
    b->tc_image = img;
    const int n_tiles = b->tile_off[b->n_frames];
    b->tc_bytes = ((size_t)n_tiles + 1) * (img == TcImage::Tf32x3 ? (size_t)kTcTileBytes : (size_t)kTc8TileBytes);
    if (img == TcImage::H) b->tc_bytes += ((size_t)b->row_off[b->n_frames] + b->n_frames) * sizeof(float);
    if (!b->d_tc || b->tc_cap < b->tc_bytes) {
        if (b->d_tc) cudaFreeAsync(b->d_tc, ctx->stream);   // (stream-ordered: earlier sweeps have been enqueued before)
        b->d_tc = nullptr;
        cudaError_t e = pool_malloc(ctx, (void**)&b->d_tc, b->tc_bytes);
        if (e != cudaSuccess) { cudaGetLastError(); return fail(ESFM_ERR_NOMEM, "cudaMallocAsync(%zu) for the tensor-core bank failed: %s", b->tc_bytes, cudaGetErrorString(e)); }
        b->tc_cap = b->tc_bytes;
    }
    cudaError_t e =
        img == TcImage::H ? launch_pack_tch((const float*)b->d_rows, b->d_frame_rows, b->d_row_off, b->d_tile_off, b->n_frames, n_tiles, b->d_tc,
                                            tch_row_eps(b), tch_frame_norm(b), ctx->stream)
        : img == TcImage::Tf32x3 ? launch_pack_tc((const float*)b->d_rows, b->d_frame_rows, b->d_row_off, b->d_tile_off, b->n_frames, n_tiles, b->d_tc, ctx->stream)
        : launch_pack_tc8((const uint32_t*)b->d_rows, b->d_frame_rows, b->d_row_off, b->d_tile_off, b->n_frames, n_tiles, b->d_tc,
                          img == TcImage::Fp8Z ? 1 : 0, ctx->stream);
    if (e != cudaSuccess) return fail(ESFM_ERR_CUDA, "tensor-core pack kernel launch failed: %s", cudaGetErrorString(e));
    if (n_tiles > 0) ctx->stats.kernel_launches += 1;
    b->tc_built = true;
    return ESFM_OK;
}

int units_per_pair(const esfm_ctx* ctx, const esfm_bank* b, const SweepPlan& sw, size_t n_chunk_pairs) {
    if (n_chunk_pairs >= (size_t)4 * ctx->sm_count) return 1;
    const int qblock_rows = sw.sweep == SweepKind::Ffma ? kQTiles * kTile : (sw.sweep == SweepKind::Popc ? kConsumerThreads * kHamRQ : kTile);
    const int max_blocks = std::max(1, (b->max_rows + qblock_rows - 1) / qblock_rows);
    const int want = (int)((4 * (size_t)ctx->sm_count + n_chunk_pairs - 1) / std::max<size_t>(n_chunk_pairs, 1));
    return std::max(1, std::min(want, max_blocks));
}

// Enqueues sweep + finalize for one chunk that is already described in cb.d_pairs (compute stream only).
int run_chunk(esfm_ctx* ctx, esfm_bank* b, const SweepPlan& sw, const ChunkPlan& pl, ChunkBuf& cb, size_t n, double ratio, int cross_check,
              int32_t* knn_idx, float* knn_dist) {
    CUDA_TRY(cudaMemsetAsync(ctx->keys, (int)(kKeyInit & 0xff), n * 4 * (size_t)pl.stride * sizeof(u64), ctx->stream));
    CUDA_TRY(cudaMemsetAsync(cb.d_cursor, 0, 4 * sizeof(unsigned long long), ctx->stream));
    if (sw.sweep == SweepKind::Tc || sw.sweep == SweepKind::Win) { if (int rc = ensure_tc_layout(ctx, b, sw.image)) return rc; }
    else if (sw.sweep == SweepKind::Ffma) { if (int rc = ensure_kmajor_layout(ctx, b)) return rc; }
    if (sw.thr_fill >= 0)
        CUDA_TRY(cudaMemsetAsync(ctx->col_thr, sw.thr_fill, n * (size_t)pl.stride * sizeof(uint32_t), ctx->stream));
    SweepParams sp{};
    sp.kmajor = b->d_kmajor;
    sp.rows_f32 = (const float*)b->d_rows;
    sp.tc_main = b->d_tc;
    sp.rows_b256 = (const uint4*)b->d_rows;
    sp.frame_rows = b->d_frame_rows;
    sp.frame_row_off = b->d_row_off;
    sp.frame_tile_off = b->d_tile_off;
    sp.pairs = cb.d_pairs;
    sp.n_pairs = (int)n;
    sp.units_per_pair = units_per_pair(ctx, b, sw, n);
    sp.keys = ctx->keys;
    sp.col_thr = ctx->col_thr;
    sp.stride = pl.stride;
    sp.col_cap = pl.col_cap;
    sp.need_cols = ((cross_check && !sw.two_phase) || knn_idx) ? 1 : 0;
    if (const char* dbg = getenv("ESFM_TC_DEBUG")) sp.debug_flags = atoi(dbg);
    sp.tc_kind = sw.image == TcImage::Fp8Z ? kTcKindB256Z : b->kind;
    sp.win_fast = sw.fast ? 1 : 0;
    if (ctx->profiling) CUDA_TRY(cudaEventRecord(cb.ev_t0, ctx->stream));
    cudaError_t e = sw.sweep == SweepKind::Win ? launch_sweep_win(sp, ctx->sm_count, ctx->stream)
                  : sw.sweep == SweepKind::Tc ? launch_sweep_l2_tc(sp, ctx->sm_count, ctx->stream)
                  : sw.sweep == SweepKind::Ffma ? launch_sweep_l2(sp, ctx->sm_count, ctx->stream)
                                                : launch_sweep_hamming(sp, ctx->sm_count, ctx->stream);
    if (e != cudaSuccess) return fail(ESFM_ERR_CUDA, "sweep kernel launch failed: %s", cudaGetErrorString(e));
    FinalizeParams fp{};
    fp.kind = b->kind;
    fp.rows_f32 = (const float*)b->d_rows;
    fp.rows_b256 = (const uint4*)b->d_rows;
    fp.frame_rows = b->d_frame_rows;
    fp.frame_row_off = b->d_row_off;
    fp.pairs = cb.d_pairs;
    fp.n_pairs = (int)n;
    fp.keys = ctx->keys;
    fp.stride = pl.stride;
    fp.ratio = ratio;
    fp.cross_check = cross_check ? 1 : 0;
    fp.key_format = sw.key_format;
    fp.phase = sw.two_phase ? 1 : 0;
    fp.gather = reinterpret_cast<int*>(ctx->col_thr);
    fp.gather_cnt = ctx->gather_cnt;
    fp.verified_rows = cb.d_cursor + 3;
    fp.arena = cb.arena;
    fp.arena_cap = cb.arena_cap;
    fp.cursor = cb.d_cursor;
    fp.overflow = (int*)(cb.d_cursor + 1);
    fp.pair_off = cb.d_pair_off;
    fp.pair_cnt = cb.d_pair_cnt;
    fp.knn_idx = knn_idx;
    fp.knn_dist = knn_dist;
    if (sw.sweep == SweepKind::Win && b->kind == ESFM_KIND_F32X64) fp.frame_norm = tch_frame_norm(b);   // (phase 1's margin, both modes)
    if (sw.fast) {
        // rows the fast sweep cannot settle -> the pair's gather list -> one exact sweep of just those rows (sweep time)
        fp.row_eps = tch_row_eps(b);
        fp.fallback_rows = cb.d_cursor + 2;
        e = launch_win_classify(fp, ctx->stream);
        if (e != cudaSuccess) return fail(ESFM_ERR_CUDA, "fast-sweep classification kernel launch failed: %s", cudaGetErrorString(e));
        SweepParams xp = sp;
        xp.win_fast = 0;
        xp.gather = fp.gather;
        xp.gather_cnt = fp.gather_cnt;
        xp.fallback = 1;
        e = launch_sweep_win(xp, ctx->sm_count, ctx->stream);
        if (e != cudaSuccess) return fail(ESFM_ERR_CUDA, "fallback sweep launch failed: %s", cudaGetErrorString(e));
        ctx->stats.kernel_launches += 2;
    }
    if (ctx->profiling) CUDA_TRY(cudaEventRecord(cb.ev_t1, ctx->stream));
    e = launch_finalize(fp, ctx->stream);
    if (e != cudaSuccess) return fail(ESFM_ERR_CUDA, "finalize kernel launch failed: %s", cudaGetErrorString(e));
    cb.two_phase = sw.two_phase;
    if (sw.two_phase) {
        SweepParams vp = sp;
        vp.gather = fp.gather;
        vp.gather_cnt = fp.gather_cnt;
        vp.win_fast = 0;
        if (ctx->profiling) CUDA_TRY(cudaEventRecord(cb.ev_v0, ctx->stream));
        e = launch_sweep_win(vp, ctx->sm_count, ctx->stream);
        if (e != cudaSuccess) return fail(ESFM_ERR_CUDA, "verification sweep launch failed: %s", cudaGetErrorString(e));
        if (ctx->profiling) CUDA_TRY(cudaEventRecord(cb.ev_v1, ctx->stream));
        fp.phase = 2;
        e = launch_finalize(fp, ctx->stream);
        if (e != cudaSuccess) return fail(ESFM_ERR_CUDA, "finalize (phase 2) kernel launch failed: %s", cudaGetErrorString(e));
        ctx->stats.kernel_launches += 2;      // (sweep_launches counts chunks swept: the verification sweep's time is added to its chunk's)
    }
    CUDA_TRY(cudaEventRecord(cb.ev_t2, ctx->stream));
    ctx->stats.kernel_launches += 2;
    ctx->stats.sweep_launches += 1;
    cb.generation += 1;
    return ESFM_OK;
}

int collect_timing(esfm_ctx* ctx, ChunkBuf& cb) {
    if (!ctx->profiling) return ESFM_OK;
    float a = 0.f, c = 0.f;
    CUDA_TRY(cudaEventElapsedTime(&a, cb.ev_t0, cb.ev_t1));
    CUDA_TRY(cudaEventElapsedTime(&c, cb.ev_t1, cb.ev_t2));
    if (cb.two_phase) {       // the verification sweep counts as sweep time, the two finalize launches as finalize time
        float v = 0.f;
        CUDA_TRY(cudaEventElapsedTime(&v, cb.ev_v0, cb.ev_v1));
        a += v;
        c -= v;
    }
    ctx->stats.last_sweep_ms = a;
    ctx->stats.last_finalize_ms = c;
    ctx->stats.sweep_ms_total += a;
    return ESFM_OK;
}

struct ResultsGuard {        // frees the half-built batch on every early return
    esfm_results* r;
    ~ResultsGuard() { if (r) esfm_results_destroy(r); }
};

void build_index(esfm_results* r) {
    if (!r->index.empty() || r->pairs.empty()) return;
    r->index.reserve(r->pairs.size() * 2);
    for (size_t k = 0; k < r->pairs.size(); ++k) {
        const uint64_t key = ((uint64_t)(uint32_t)r->pairs[k].q_frame << 32) | (uint32_t)r->pairs[k].t_frame;
        r->index.emplace(key, (int64_t)k);
    }
}

constexpr uint64_t kOffMask = ((uint64_t)1 << 40) - 1;

}  // namespace

// The chunk pipeline.  Chunk k is swept and finalised on the compute stream into arena[k & 1]; its per-pair counts and
// offsets, then its matches, travel to the host on the copy stream while chunk k + 1 is being swept; the host thread stays one
// chunk ahead of the device:
//     iteration k:  enqueue compute(k) | finish(k-1): wait for counts(k-1), bring its matches to the host | enqueue counts(k)
// A one-chunk batch lands in ONE pinned buffer borrowed from the context's pool (kept by the results; steady-state calls reuse
// it); the chunks of a longer batch are streamed through small pinned slots into pageable, huge-page-advised segments.
int esfm::match_pairs_impl(esfm_bank* b, const esfm_pair_t* pairs, int64_t n_pairs, double ratio, int cross_check, const MatchOpts& opts,
                           esfm_results** out) {
    if (!b || !out) return fail(ESFM_ERR_INVALID, "esfm_match_pairs: NULL argument");
    *out = nullptr;
    if (!b->committed) return fail(ESFM_ERR_STATE, "esfm_match_pairs: bank not committed");
    if (n_pairs < 0 || (n_pairs > 0 && !pairs)) return fail(ESFM_ERR_INVALID, "esfm_match_pairs: bad pair list");
    if (!(ratio == ratio)) return fail(ESFM_ERR_INVALID, "ratio is NaN");
    if (opts.keep != ESFM_KEEP_MATCHES && opts.keep != ESFM_KEEP_DIGESTS) return fail(ESFM_ERR_INVALID, "unknown keep mode %d", opts.keep);
    esfm_ctx* ctx = b->ctx;
    if (int rc = set_device(ctx)) return rc;
    for (int64_t k = 0; k < n_pairs; ++k)
        if (pairs[k].query < 0 || pairs[k].query >= b->n_frames || pairs[k].train < 0 || pairs[k].train >= b->n_frames)
            return fail(ESFM_ERR_INVALID, "pair %lld = (%d,%d) out of range [0,%d)", (long long)k, pairs[k].query, pairs[k].train, b->n_frames);

    esfm_results* res = new (std::nothrow) esfm_results();
    if (!res) return fail(ESFM_ERR_NOMEM, "out of host memory");
    ResultsGuard guard{res};
    const bool digests_only = opts.fetch && opts.keep == ESFM_KEEP_DIGESTS;
    res->ctx = ctx;
    res->kind = b->kind;
    res->ratio = ratio;
    res->cross_check = cross_check ? 1 : 0;
    res->keep = opts.keep;
    res->frame_rows.assign(b->rows.begin(), b->rows.end());
    res->pairs.resize((size_t)n_pairs);
    res->counts.assign((size_t)n_pairs, 0);
    res->offsets.assign((size_t)n_pairs, 0);
    if (digests_only) res->digests.assign((size_t)n_pairs, 0);
    res->fetched = opts.fetch;
    for (int64_t k = 0; k < n_pairs; ++k) {
        res->pairs[(size_t)k].q_frame = pairs[k].query;
        res->pairs[(size_t)k].t_frame = pairs[k].train;
    }
    if (n_pairs == 0) { guard.r = nullptr; *out = res; return ESFM_OK; }

    const SweepPlan sw = plan_sweep(ctx, b, cross_check != 0, false);
    const ChunkPlan pl = plan_chunks(b, n_pairs);
    const size_t n_chunks = ((size_t)n_pairs + pl.chunk_pairs - 1) / pl.chunk_pairs;
    const bool streamed = opts.fetch && (n_chunks > 1 || digests_only);   // matches go to pageable memory through the pinned slots
    if (int rc = ensure_scratch(ctx, b, sw, pl, n_chunks > 1 ? 2 : 1)) return rc;

    struct Chunk { size_t c0 = 0, n = 0; std::vector<uint32_t> order; };
    Chunk chunks[2];

    auto enqueue_compute = [&](size_t k) -> int {
        Chunk& ch = chunks[k & 1];
        ChunkBuf& cb = ctx->buf[k & 1];
        ch.c0 = k * pl.chunk_pairs;
        ch.n = std::min(pl.chunk_pairs, (size_t)n_pairs - ch.c0);
        // Launch order inside the chunk: by TRAIN frame.  The sweep re-streams the train frame once per query block
        // (32x per pair at 8k rows), the query frame only once; CTAs that run concurrently take consecutive units, so
        // sorting by train frame makes them stream the SAME tiles and L2 serves the re-reads (the reference's loop order
        // shares the query frame instead and cost 6-15x the algorithmic DRAM traffic, profiles/traffic_bench_r1.csv).
        ch.order.resize(ch.n);
        for (size_t i = 0; i < ch.n; ++i) ch.order[i] = (uint32_t)i;
        const PairDesc* pp = res->pairs.data() + ch.c0;
        std::stable_sort(ch.order.begin(), ch.order.end(), [pp](uint32_t a, uint32_t b2) {
            return pp[a].t_frame != pp[b2].t_frame ? pp[a].t_frame < pp[b2].t_frame : pp[a].q_frame < pp[b2].q_frame;
        });
        for (size_t i = 0; i < ch.n; ++i) cb.h_pairs[i] = pp[ch.order[i]];
        if (cb.copy_pending) {        // the download of the chunk that used this arena two iterations ago
            CUDA_TRY(cudaStreamWaitEvent(ctx->stream, cb.ev_copied, 0));
            cb.copy_pending = false;
        }
        CUDA_TRY(cudaMemcpyAsync(cb.d_pairs, cb.h_pairs, ch.n * sizeof(PairDesc), cudaMemcpyHostToDevice, ctx->stream));
        ctx->stats.h2d_bytes += ch.n * sizeof(PairDesc);
        return run_chunk(ctx, b, sw, pl, cb, ch.n, ratio, cross_check, nullptr, nullptr);
    };
    auto enqueue_meta = [&](size_t k) -> int {      // counts + offsets + cursor of chunk k -> pinned host memory (copy stream)
        Chunk& ch = chunks[k & 1];
        ChunkBuf& cb = ctx->buf[k & 1];
        CUDA_TRY(cudaStreamWaitEvent(ctx->copy_stream, cb.ev_t2, 0));
        unsigned long long* h_cur = (unsigned long long*)cb.h_meta;
        unsigned long long* h_off = h_cur + 4;
        int32_t* h_cnt = (int32_t*)(h_off + ch.n);
        CUDA_TRY(cudaMemcpyAsync(h_cur, cb.d_cursor, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, ctx->copy_stream));
        CUDA_TRY(cudaMemcpyAsync(h_off, cb.d_pair_off, ch.n * sizeof(unsigned long long), cudaMemcpyDeviceToHost, ctx->copy_stream));
        CUDA_TRY(cudaMemcpyAsync(h_cnt, cb.d_pair_cnt, ch.n * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->copy_stream));
        CUDA_TRY(cudaEventRecord(cb.ev_meta, ctx->copy_stream));
        ctx->stats.d2h_bytes += ch.n * (sizeof(int32_t) + sizeof(unsigned long long)) + 4 * sizeof(unsigned long long);
        return ESFM_OK;
    };
    auto finish = [&](size_t k) -> int {            // chunk k has been finalised: book its pairs, bring its matches to the host
        Chunk& ch = chunks[k & 1];
        ChunkBuf& cb = ctx->buf[k & 1];
        CUDA_TRY(cudaEventSynchronize(cb.ev_meta));
        if (int rc = collect_timing(ctx, cb)) return rc;
        const unsigned long long* h_cur = (const unsigned long long*)cb.h_meta;
        const unsigned long long* h_off = h_cur + 4;
        const int32_t* h_cnt = (const int32_t*)(h_off + ch.n);
        const unsigned long long n_matches = h_cur[0];
        if ((int)h_cur[1] != 0 || n_matches > cb.arena_cap) return fail(ESFM_ERR_CAPACITY, "match arena overflow (internal sizing error)");
        ctx->stats.fallback_rows += h_cur[2];
        ctx->stats.verified_rows += h_cur[3];
        const int seg = (int)res->segments.size();
        for (size_t i = 0; i < ch.n; ++i) {
            res->counts[ch.c0 + ch.order[i]] = h_cnt[i];
            res->offsets[ch.c0 + ch.order[i]] = ((uint64_t)seg << 40) | (uint64_t)h_off[i];
            const PairDesc& pd = cb.h_pairs[i];
            ctx->stats.comparisons += (uint64_t)b->rows[pd.q_frame] * (uint64_t)b->rows[pd.t_frame];
        }
        ctx->stats.pairs += ch.n;
        res->total_matches += (int64_t)n_matches;
        if (!opts.fetch) {
            res->dev_buf = (int)(k & 1);
            res->device_matches = n_matches;
            res->arena_generation = n_chunks > 1 ? 0 : cb.generation;   // several chunks: the arenas are reused, nothing to fetch later
            return ESFM_OK;
        }
        const size_t bytes = (size_t)n_matches * sizeof(esfm_dmatch_t);
        if (!streamed) {
            esfm_results::Segment sg{nullptr, (size_t)n_matches, ctx};
            if (n_matches > 0) {
                sg.ptr = (esfm_dmatch_t*)pool_acquire(ctx, bytes, nullptr);
                if (!sg.ptr) return fail(ESFM_ERR_NOMEM, "pinned buffer of %zu bytes for the matches failed", bytes);
            }
            res->segments.push_back(sg);
            if (n_matches > 0) {
                CUDA_TRY(cudaMemcpyAsync(sg.ptr, cb.arena, bytes, cudaMemcpyDeviceToHost, ctx->copy_stream));
                ctx->stats.d2h_bytes += bytes;
                CUDA_TRY(cudaStreamSynchronize(ctx->copy_stream));
            }
            return ESFM_OK;
        }
        esfm_dmatch_t* dst = nullptr;
        if (digests_only) {
            if (ctx->h_scratch_cap < (size_t)n_matches) {
                free(ctx->h_scratch);
                ctx->h_scratch_cap = 0;
                const size_t want = (size_t)n_matches + (size_t)n_matches / 4;
                ctx->h_scratch = heap_segment_alloc(want);
                if (!ctx->h_scratch) return fail(ESFM_ERR_NOMEM, "host scratch of %zu bytes failed", want * sizeof(esfm_dmatch_t));
                ctx->h_scratch_cap = want;
            }
            dst = ctx->h_scratch;
        } else {
            esfm_results::Segment sg{nullptr, (size_t)n_matches, nullptr};
            if (n_matches > 0) {
                sg.ptr = heap_segment_alloc((size_t)n_matches);
                if (!sg.ptr) return fail(ESFM_ERR_NOMEM, "host buffer of %zu bytes for the matches failed", bytes);
            }
            res->segments.push_back(sg);
            dst = sg.ptr;
        }
        if (n_matches > 0)
            if (int rc = stream_down(ctx, cb.arena, dst, (size_t)n_matches)) return rc;
        // every piece has left the arena: the chunk after next may overwrite it
        CUDA_TRY(cudaEventRecord(cb.ev_copied, ctx->copy_stream));
        cb.copy_pending = true;
        if (digests_only) {
            // the digests of a chunk's pairs are independent: a few helper threads share them (one thread digests ~3 GB/s, and the
            // 12.5 M-pair ORB job returns 25 GB of matches per device: the host was the bottleneck of the whole job)
            auto digest_range = [&](size_t i0, size_t i1) {
                for (size_t i = i0; i < i1; ++i) {
                    const size_t g = ch.c0 + ch.order[i];
                    res->digests[g] = digest_matches(dst + (res->offsets[g] & kOffMask), res->counts[g]);
                }
            };
            int helpers = 4;
            if (const char* e = getenv("ESFM_COPY_THREADS")) helpers = std::max(1, std::min(16, atoi(e)));
            if (helpers <= 1 || n_matches < (1 << 20)) digest_range(0, ch.n);
            else {
                std::vector<std::thread> th;
                const size_t per = (ch.n + (size_t)helpers - 1) / (size_t)helpers;
                for (int t = 1; t < helpers; ++t) {
                    const size_t i0 = std::min(ch.n, per * (size_t)t), i1 = std::min(ch.n, per * (size_t)(t + 1));
                    if (i0 < i1) th.emplace_back(digest_range, i0, i1);
                }
                digest_range(0, std::min(ch.n, per));
                for (auto& t : th) t.join();
            }
        }
        return ESFM_OK;
    };

    int rc = ESFM_OK;
    for (size_t k = 0; k < n_chunks && !rc; ++k) {
        rc = enqueue_compute(k);
        if (!rc && k >= 1) rc = finish(k - 1);      // (the device is busy with chunk k meanwhile)
        if (!rc) rc = enqueue_meta(k);
    }
    if (!rc) rc = finish(n_chunks - 1);
    if (rc) {
        cudaStreamSynchronize(ctx->stream);         // nothing may still write into buffers the guard is about to release
        cudaStreamSynchronize(ctx->copy_stream);
        return rc;
    }
    guard.r = nullptr;
    *out = res;
    return ESFM_OK;
}

extern "C" int esfm_match_pairs(esfm_bank_t* b, const esfm_pair_t* pairs, int64_t n_pairs, double ratio, int cross_check,
                                esfm_results_t** results) {
    return match_pairs_impl(b, pairs, n_pairs, ratio, cross_check, MatchOpts{true, ESFM_KEEP_MATCHES}, results);
}

extern "C" int esfm_match_pairs_keep(esfm_bank_t* b, const esfm_pair_t* pairs, int64_t n_pairs, double ratio, int cross_check, int keep,
                                     esfm_results_t** results) {
    return match_pairs_impl(b, pairs, n_pairs, ratio, cross_check, MatchOpts{true, keep}, results);
}

extern "C" int esfm_match_pairs_device(esfm_bank_t* b, const esfm_pair_t* pairs, int64_t n_pairs, double ratio,
                                       int cross_check, esfm_results_t** results) {
    return match_pairs_impl(b, pairs, n_pairs, ratio, cross_check, MatchOpts{false, ESFM_KEEP_MATCHES}, results);
}

extern "C" int esfm_bank_chunk_pairs(esfm_bank_t* b, int64_t* max_pairs) {
    if (!b || !max_pairs) return fail(ESFM_ERR_INVALID, "esfm_bank_chunk_pairs: NULL argument");
    if (!b->committed) return fail(ESFM_ERR_STATE, "bank not committed");
    *max_pairs = (int64_t)plan_chunks(b, (int64_t)1 << 40).chunk_pairs;
    return ESFM_OK;
}

static int device_batch_check(esfm_results* r) {
    if (!r) return fail(ESFM_ERR_INVALID, "results is NULL");
    if (r->fetched && r->arena_generation == 0) return fail(ESFM_ERR_STATE, "not a device-resident batch");
    if (!r->ctx || r->arena_generation == 0 || r->arena_generation != r->ctx->buf[r->dev_buf].generation)
        return fail(ESFM_ERR_STATE, "device-resident matches are gone (the arena was reused by a later batch or the batch spanned several chunks)");
    return ESFM_OK;
}

extern "C" int esfm_results_fetch(esfm_results_t* r) {
    if (!r) return fail(ESFM_ERR_INVALID, "results is NULL");
    if (r->fetched) return ESFM_OK;
    if (int rc = device_batch_check(r)) return rc;
    esfm_ctx* ctx = r->ctx;
    if (int rc = set_device(ctx)) return rc;
    esfm_results::Segment sg{nullptr, (size_t)r->device_matches, ctx};
    if (r->device_matches > 0) {
        const size_t bytes = (size_t)r->device_matches * sizeof(esfm_dmatch_t);
        sg.ptr = (esfm_dmatch_t*)pool_acquire(ctx, bytes, nullptr);
        if (!sg.ptr) return fail(ESFM_ERR_NOMEM, "pinned buffer of %zu bytes for the matches failed", bytes);
        cudaError_t e = cudaMemcpyAsync(sg.ptr, ctx->buf[r->dev_buf].arena, bytes, cudaMemcpyDeviceToHost, ctx->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess) { pool_release(ctx, sg.ptr); return fail(ESFM_ERR_CUDA, "match download failed: %s", cudaGetErrorString(e)); }
        ctx->stats.d2h_bytes += bytes;
    }
    r->segments.assign(1, sg);
    r->fetched = true;
    return ESFM_OK;
}

extern "C" int esfm_results_device_matches(esfm_results_t* r, void** dev_ptr, int64_t* n_matches) {
    if (!dev_ptr || !n_matches) return fail(ESFM_ERR_INVALID, "esfm_results_device_matches: NULL argument");
    if (int rc = device_batch_check(r)) return rc;
    *dev_ptr = r->ctx->buf[r->dev_buf].arena;
    *n_matches = (int64_t)r->device_matches;
    return ESFM_OK;
}

extern "C" int esfm_results_device_layout(esfm_results_t* r, int64_t* offsets) {
    if (!r || !offsets) return fail(ESFM_ERR_INVALID, "esfm_results_device_layout: NULL argument");
    for (size_t k = 0; k < r->pairs.size(); ++k) offsets[k] = (int64_t)(r->offsets[k] & kOffMask);
    return ESFM_OK;
}

extern "C" int esfm_match_all_pairs(esfm_bank_t* b, double ratio, int cross_check, esfm_results_t** results) {
    if (!b || !results) return fail(ESFM_ERR_INVALID, "esfm_match_all_pairs: NULL argument");
    std::vector<esfm_pair_t> pairs;
    const int n = b->n_frames;
    pairs.reserve((size_t)n * (size_t)(n > 0 ? n - 1 : 0) / 2);
    for (int i = 0; i < n; ++i)           // cpp_code/test/sfm.cpp:140
        for (int j = 0; j < i; ++j) {     // cpp_code/test/sfm.cpp:143
            esfm_pair_t p;
            p.query = i;                  // frames[i] is cur_frame_1 = query  (sfm.cpp:153,156)
            p.train = j;
            pairs.push_back(p);
        }
    return match_pairs_impl(b, pairs.data(), (int64_t)pairs.size(), ratio, cross_check, MatchOpts{true, ESFM_KEEP_MATCHES}, results);
}

extern "C" int esfm_match_pair(esfm_bank_t* b, int query_frame, int train_frame, double ratio, int cross_check,
                               esfm_dmatch_t* out, int cap, int* n_matches) {
    if (!n_matches) return fail(ESFM_ERR_INVALID, "n_matches is NULL");
    *n_matches = 0;
    esfm_pair_t p;
    p.query = query_frame;
    p.train = train_frame;
    esfm_results* r = nullptr;
    if (int rc = match_pairs_impl(b, &p, 1, ratio, cross_check, MatchOpts{true, ESFM_KEEP_MATCHES}, &r)) return rc;
    const int n = r->counts[0];
    if (n > cap || (n > 0 && !out)) {
        esfm_results_destroy(r);
        return fail(ESFM_ERR_CAPACITY, "output buffer holds %d matches, %d needed", cap, n);
    }
    if (n > 0) memcpy(out, r->segments[0].ptr + (r->offsets[0] & kOffMask), (size_t)n * sizeof(esfm_dmatch_t));
    *n_matches = n;
    esfm_results_destroy(r);
    return ESFM_OK;
}

// The unmodified caller's shape (sfm.cpp:153,156 -> matchFeaturesX(frame_i, frame_j, ...)): one pair per call.  The context
// keeps ONE two-frame bank per kind and refills it, so a call costs two staged uploads, one pack kernel, sweep + finalize
// and the match download -- no device allocation once the largest frame pair has been seen.
extern "C" int esfm_match_descriptors(esfm_ctx_t* ctx, esfm_kind kind, const void* query, int rows_q, size_t step_q,
                                      const void* train, int rows_t, size_t step_t, int cols, double ratio, int cross_check,
                                      esfm_dmatch_t* out, int cap, int* n_matches) {
    if (!n_matches) return fail(ESFM_ERR_INVALID, "n_matches is NULL");
    *n_matches = 0;
    if (!ctx) return fail(ESFM_ERR_INVALID, "ctx is NULL");
    if (kind != ESFM_KIND_F32X64 && kind != ESFM_KIND_B256) return fail(ESFM_ERR_INVALID, "esfm_match_descriptors: unknown kind %d", (int)kind);
    esfm_bank*& b = ctx->pair_bank[kind];
    if (!b) {
        if (int rc = esfm_bank_create(ctx, kind, 2, &b)) return rc;
    } else {
        bank_reset(b);
    }
    int rc = esfm_bank_set_frame(b, 0, query, rows_q, cols, step_q);
    if (!rc) rc = esfm_bank_set_frame(b, 1, train, rows_t, cols, step_t);
    if (!rc) rc = esfm_bank_commit(b);
    if (!rc) rc = esfm_match_pair(b, 0, 1, ratio, cross_check, out, cap, n_matches);
    if (rc) {               // leave no half-filled bank behind
        esfm_bank_destroy(b);
        b = nullptr;
    }
    return rc;
}

extern "C" int esfm_knn2_pair(esfm_bank_t* b, int query_frame, int train_frame, int32_t* idx, float* dist) {
    if (!b || !idx || !dist) return fail(ESFM_ERR_INVALID, "esfm_knn2_pair: NULL argument");
    if (!b->committed) return fail(ESFM_ERR_STATE, "bank not committed");
    if (query_frame < 0 || query_frame >= b->n_frames || train_frame < 0 || train_frame >= b->n_frames)
        return fail(ESFM_ERR_INVALID, "frame index out of range");
    esfm_ctx* ctx = b->ctx;
    if (int rc = set_device(ctx)) return rc;
    const int fq = b->rows[query_frame];
    if (fq == 0) return ESFM_OK;
    const SweepPlan sw = plan_sweep(ctx, b, false, true);
    const ChunkPlan pl = plan_chunks(b, 1);
    if (int rc = ensure_scratch(ctx, b, sw, pl, 1)) return rc;
    ChunkBuf& cb = ctx->buf[0];
    int32_t* d_idx = nullptr;
    float* d_dist = nullptr;
    CUDA_TRY(cudaMalloc((void**)&d_idx, (size_t)fq * 2 * sizeof(int32_t)));
    cudaError_t e = cudaMalloc((void**)&d_dist, (size_t)fq * 2 * sizeof(float));
    if (e != cudaSuccess) { cudaFree(d_idx); return fail(ESFM_ERR_NOMEM, "cudaMalloc failed: %s", cudaGetErrorString(e)); }
    cb.h_pairs[0].q_frame = query_frame;
    cb.h_pairs[0].t_frame = train_frame;
    int rc = ESFM_OK;
    e = cudaMemcpyAsync(cb.d_pairs, cb.h_pairs, sizeof(PairDesc), cudaMemcpyHostToDevice, ctx->stream);
    if (e != cudaSuccess) rc = fail(ESFM_ERR_CUDA, "cudaMemcpyAsync failed: %s", cudaGetErrorString(e));
    if (!rc) rc = run_chunk(ctx, b, sw, pl, cb, 1, 0.0, 0, d_idx, d_dist);
    if (!rc) {
        e = cudaMemcpyAsync(idx, d_idx, (size_t)fq * 2 * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(dist, d_dist, (size_t)fq * 2 * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess) rc = fail(ESFM_ERR_CUDA, "knn2 copy back failed: %s", cudaGetErrorString(e));
        ctx->stats.d2h_bytes += (size_t)fq * 16;
        ctx->stats.pairs += 1;
        ctx->stats.comparisons += (uint64_t)fq * (uint64_t)b->rows[train_frame];
    }
    cudaFree(d_idx);
    cudaFree(d_dist);
    if (!rc) rc = collect_timing(ctx, cb);
    return rc;
}

// ------------------------------------------------------------------------------------------------
// results
// ------------------------------------------------------------------------------------------------
extern "C" int esfm_results_counts(esfm_results_t* r, int64_t* n_pairs, int64_t* n_matches) {
    if (!r) return fail(ESFM_ERR_INVALID, "results is NULL");
    if (n_pairs) *n_pairs = (int64_t)r->pairs.size();
    if (n_matches) *n_matches = r->total_matches;
    return ESFM_OK;
}

static const esfm_dmatch_t* pair_ptr(const esfm_results* r, size_t k) {
    const uint64_t o = r->offsets[k];
    return r->counts[k] > 0 ? r->segments[(size_t)(o >> 40)].ptr + (o & kOffMask) : nullptr;
}

extern "C" int esfm_results_pair_at(esfm_results_t* r, int64_t k, int* query_frame, int* train_frame,
                                    const esfm_dmatch_t** matches, int* n_matches) {
    if (!r) return fail(ESFM_ERR_INVALID, "results is NULL");
    if (k < 0 || k >= (int64_t)r->pairs.size()) return fail(ESFM_ERR_INVALID, "pair index %lld out of range", (long long)k);
    if (query_frame) *query_frame = r->pairs[(size_t)k].q_frame;
    if (train_frame) *train_frame = r->pairs[(size_t)k].t_frame;
    if (n_matches) *n_matches = r->counts[(size_t)k];
    if (matches) {
        if (!r->fetched) return fail(ESFM_ERR_STATE, "matches are device-resident; call esfm_results_fetch first");
        if (r->keep == ESFM_KEEP_DIGESTS) return fail(ESFM_ERR_STATE, "this batch kept per-pair digests only (ESFM_KEEP_DIGESTS)");
        *matches = pair_ptr(r, (size_t)k);
    }
    return ESFM_OK;
}

extern "C" int esfm_results_pair(esfm_results_t* r, int query_frame, int train_frame, const esfm_dmatch_t** matches,
                                 int* n_matches) {
    if (!r) return fail(ESFM_ERR_INVALID, "results is NULL");
    build_index(r);
    const uint64_t key = ((uint64_t)(uint32_t)query_frame << 32) | (uint32_t)train_frame;
    auto it = r->index.find(key);
    if (it == r->index.end()) return fail(ESFM_ERR_INVALID, "pair (%d,%d) is not part of this batch", query_frame, train_frame);
    return esfm_results_pair_at(r, it->second, nullptr, nullptr, matches, n_matches);
}

extern "C" int esfm_results_pair_counts(esfm_results_t* r, int32_t* counts) {
    if (!r || !counts) return fail(ESFM_ERR_INVALID, "NULL argument");
    if (!r->counts.empty()) memcpy(counts, r->counts.data(), r->counts.size() * sizeof(int32_t));
    return ESFM_OK;
}

extern "C" int esfm_results_copy_all(esfm_results_t* r, esfm_dmatch_t* out, int64_t cap, int64_t* offsets) {
    if (!r) return fail(ESFM_ERR_INVALID, "results is NULL");
    if (!r->fetched) return fail(ESFM_ERR_STATE, "matches are device-resident; call esfm_results_fetch first");
    if (r->keep == ESFM_KEEP_DIGESTS) return fail(ESFM_ERR_STATE, "this batch kept per-pair digests only (ESFM_KEEP_DIGESTS)");
    if (cap < r->total_matches || (r->total_matches > 0 && !out)) return fail(ESFM_ERR_CAPACITY, "output holds %lld matches, %lld needed", (long long)cap, (long long)r->total_matches);
    int64_t pos = 0;
    for (size_t k = 0; k < r->pairs.size(); ++k) {
        if (offsets) offsets[k] = pos;
        const int32_t n = r->counts[k];
        if (n > 0) memcpy(out + pos, pair_ptr(r, k), (size_t)n * sizeof(esfm_dmatch_t));
        pos += n;
    }
    if (offsets) offsets[r->pairs.size()] = pos;
    return ESFM_OK;
}

static int host_batch_check(esfm_results* r) {
    if (!r) return fail(ESFM_ERR_INVALID, "results is NULL");
    if (!r->fetched) return fail(ESFM_ERR_STATE, "matches are device-resident; call esfm_results_fetch first");
    if (r->keep == ESFM_KEEP_DIGESTS) return fail(ESFM_ERR_STATE, "this batch kept per-pair digests only (ESFM_KEEP_DIGESTS)");
    return ESFM_OK;
}

extern "C" int esfm_results_segment_count(esfm_results_t* r, int* n_segments) {
    if (!n_segments) return fail(ESFM_ERR_INVALID, "esfm_results_segment_count: NULL argument");
    if (int rc = host_batch_check(r)) return rc;
    *n_segments = (int)r->segments.size();
    return ESFM_OK;
}

extern "C" int esfm_results_segment_at(esfm_results_t* r, int segment, const esfm_dmatch_t** matches, int64_t* n_matches) {
    if (!matches || !n_matches) return fail(ESFM_ERR_INVALID, "esfm_results_segment_at: NULL argument");
    if (int rc = host_batch_check(r)) return rc;
    if (segment < 0 || segment >= (int)r->segments.size()) return fail(ESFM_ERR_INVALID, "segment %d out of range [0,%zu)", segment, r->segments.size());
    *matches = r->segments[(size_t)segment].ptr;
    *n_matches = (int64_t)r->segments[(size_t)segment].count;
    return ESFM_OK;
}

extern "C" int esfm_results_pair_layout(esfm_results_t* r, int32_t* segment, int64_t* offset) {
    if (!segment || !offset) return fail(ESFM_ERR_INVALID, "esfm_results_pair_layout: NULL argument");
    if (int rc = host_batch_check(r)) return rc;
    for (size_t k = 0; k < r->pairs.size(); ++k) {
        segment[k] = (int32_t)(r->offsets[k] >> 40);
        offset[k] = (int64_t)(r->offsets[k] & kOffMask);
    }
    return ESFM_OK;
}

extern "C" int esfm_results_digests(esfm_results_t* r, uint64_t* digests) {
    if (!r || !digests) return fail(ESFM_ERR_INVALID, "esfm_results_digests: NULL argument");
    if (!r->digests.empty() || r->pairs.empty()) {
        if (!r->digests.empty()) memcpy(digests, r->digests.data(), r->digests.size() * sizeof(uint64_t));
        return ESFM_OK;
    }
    if (!r->fetched) return fail(ESFM_ERR_STATE, "matches are device-resident; call esfm_results_fetch first");
    for (size_t k = 0; k < r->pairs.size(); ++k) digests[k] = digest_matches(pair_ptr(r, k), r->counts[k]);
    return ESFM_OK;
}

extern "C" int esfm_results_destroy(esfm_results_t* r) {
    if (!r) return ESFM_OK;
    for (auto& s : r->segments) {
        if (s.pool_ctx) pool_release(s.pool_ctx, s.ptr);
        else free(s.ptr);
    }
    delete r;
    return ESFM_OK;
}

// ------------------------------------------------------------------------------------------------
// persistence of a fetched batch (host only)
// ------------------------------------------------------------------------------------------------
namespace {
struct MatchFileHeader {
    char magic[8];
    uint32_t version, dmatch_bytes;
    int64_t n_pairs, n_matches;
    int32_t kind, cross_check;
    double ratio;
};
static_assert(sizeof(MatchFileHeader) == 48, "match file header layout");
const char kMatchMagic[8] = {'E', 'S', 'F', 'M', 'M', 'T', 'C', 'H'};
}  // namespace

extern "C" int esfm_results_save(esfm_results_t* r, const char* path) {
    if (!r || !path) return fail(ESFM_ERR_INVALID, "esfm_results_save: NULL argument");
    if (!r->fetched) return fail(ESFM_ERR_STATE, "matches are device-resident; call esfm_results_fetch first");
    if (r->keep == ESFM_KEEP_DIGESTS) return fail(ESFM_ERR_STATE, "this batch kept per-pair digests only (ESFM_KEEP_DIGESTS)");
    FILE* f = fopen(path, "wb");
    if (!f) return fail(ESFM_ERR_INVALID, "esfm_results_save: cannot open %s for writing", path);
    MatchFileHeader h{};
    memcpy(h.magic, kMatchMagic, 8);
    h.version = r->frame_rows.empty() ? 1 : 2;
    h.dmatch_bytes = (uint32_t)sizeof(esfm_dmatch_t);
    h.n_pairs = (int64_t)r->pairs.size();
    h.n_matches = 0;
    for (int32_t c : r->counts) h.n_matches += c;
    h.kind = r->kind;
    h.cross_check = r->cross_check;
    h.ratio = r->ratio;
    bool ok = fwrite(&h, sizeof h, 1, f) == 1;
    if (ok && h.version == 2) {
        const int32_t nf[2] = {(int32_t)r->frame_rows.size(), 0};
        ok = fwrite(nf, sizeof nf, 1, f) == 1 && fwrite(r->frame_rows.data(), sizeof(int32_t), r->frame_rows.size(), f) == r->frame_rows.size();
    }
    static_assert(sizeof(PairDesc) == sizeof(esfm_pair_t), "pair layout");
    if (ok && h.n_pairs) ok = fwrite(r->pairs.data(), sizeof(PairDesc), r->pairs.size(), f) == r->pairs.size();
    if (ok && h.n_pairs) ok = fwrite(r->counts.data(), sizeof(int32_t), r->counts.size(), f) == r->counts.size();
    for (size_t k = 0; ok && k < r->pairs.size(); ++k) {
        const int32_t n = r->counts[k];
        if (n <= 0) continue;
        ok = fwrite(pair_ptr(r, k), sizeof(esfm_dmatch_t), (size_t)n, f) == (size_t)n;
    }
    ok = (fclose(f) == 0) && ok;
    if (!ok) return fail(ESFM_ERR_INVALID, "esfm_results_save: short write to %s", path);
    return ESFM_OK;
}

extern "C" int esfm_results_params(esfm_results_t* r, int* kind, double* ratio, int* cross_check) {
    if (!r) return fail(ESFM_ERR_INVALID, "results is NULL");
    if (kind) *kind = r->kind;
    if (ratio) *ratio = r->ratio;
    if (cross_check) *cross_check = r->cross_check;
    return ESFM_OK;
}

extern "C" int esfm_results_frame_rows(esfm_results_t* r, int32_t* rows, int cap, int* n_frames) {
    if (!r || !n_frames) return fail(ESFM_ERR_INVALID, "esfm_results_frame_rows: NULL argument");
    *n_frames = (int)r->frame_rows.size();
    if (rows) {
        if (cap < *n_frames) return fail(ESFM_ERR_CAPACITY, "rows holds %d entries, %d needed", cap, *n_frames);
        if (*n_frames) memcpy(rows, r->frame_rows.data(), r->frame_rows.size() * sizeof(int32_t));
    }
    return ESFM_OK;
}

// Does this batch belong to a frame list with these row counts?  Every pair's frame ids, the stored row counts (version-2
// files) and EVERY match index are checked: a file saved for another image set must not hand out-of-range queryIdx / trainIdx
// to the RANSAC / triangulation code that indexes frame.keypoints with them (estimate_motion.cpp:40-47).
extern "C" int esfm_results_validate(esfm_results_t* r, int n_frames, const int32_t* rows) {
    if (!r || (n_frames > 0 && !rows) || n_frames < 0) return fail(ESFM_ERR_INVALID, "esfm_results_validate: bad argument");
    if (!r->frame_rows.empty()) {
        if ((int)r->frame_rows.size() != n_frames) return fail(ESFM_ERR_INVALID, "the batch was matched on %zu frames, the caller has %d", r->frame_rows.size(), n_frames);
        for (int f = 0; f < n_frames; ++f)
            if (r->frame_rows[(size_t)f] != rows[f]) return fail(ESFM_ERR_INVALID, "frame %d had %d descriptors when the batch was matched, now %d", f, r->frame_rows[(size_t)f], rows[f]);
    }
    const bool scan = r->fetched && r->keep == ESFM_KEEP_MATCHES;
    for (size_t k = 0; k < r->pairs.size(); ++k) {
        const int q = r->pairs[k].q_frame, t = r->pairs[k].t_frame;
        if (q < 0 || q >= n_frames || t < 0 || t >= n_frames) return fail(ESFM_ERR_INVALID, "pair %zu = (%d,%d) is outside the caller's %d frames", k, q, t, n_frames);
        if (!scan) continue;
        const esfm_dmatch_t* m = pair_ptr(r, k);
        for (int32_t i = 0; i < r->counts[k]; ++i)
            if (m[i].queryIdx < 0 || m[i].queryIdx >= rows[q] || m[i].trainIdx < 0 || m[i].trainIdx >= rows[t])
                return fail(ESFM_ERR_INVALID, "pair (%d,%d): match %d = (%d,%d) is outside the frames' %d x %d descriptors", q, t, i, m[i].queryIdx, m[i].trainIdx, rows[q], rows[t]);
    }
    return ESFM_OK;
}

extern "C" int esfm_results_load(const char* path, esfm_results_t** out) {
    if (!path || !out) return fail(ESFM_ERR_INVALID, "esfm_results_load: NULL argument");
    *out = nullptr;
    FILE* f = fopen(path, "rb");
    if (!f) return fail(ESFM_ERR_INVALID, "esfm_results_load: cannot open %s", path);
    MatchFileHeader h{};
    if (fread(&h, sizeof h, 1, f) != 1 || memcmp(h.magic, kMatchMagic, 8) != 0 || (h.version != 1 && h.version != 2) ||
        h.dmatch_bytes != sizeof(esfm_dmatch_t) || h.n_pairs < 0 || h.n_matches < 0) {
        fclose(f);
        return fail(ESFM_ERR_INVALID, "esfm_results_load: %s is not an esfm match file (version 1 or 2)", path);
    }
    esfm_results* r = new (std::nothrow) esfm_results();
    if (!r) { fclose(f); return fail(ESFM_ERR_NOMEM, "out of host memory"); }
    r->fetched = true;
    r->kind = h.kind;
    r->cross_check = h.cross_check;
    r->ratio = h.ratio;
    bool ok = true;
    if (h.version == 2) {
        int32_t nf[2] = {0, 0};
        ok = fread(nf, sizeof nf, 1, f) == 1 && nf[0] >= 0 && nf[0] < (1 << 28);
        if (ok) {
            try { r->frame_rows.resize((size_t)nf[0]); } catch (...) { ok = false; }
        }
        if (ok && nf[0]) ok = fread(r->frame_rows.data(), sizeof(int32_t), r->frame_rows.size(), f) == r->frame_rows.size();
    }
    if (ok) try {
        r->pairs.resize((size_t)h.n_pairs);
        r->counts.resize((size_t)h.n_pairs);
        r->offsets.resize((size_t)h.n_pairs);
    } catch (...) { ok = false; }
    if (ok && h.n_pairs) ok = fread(r->pairs.data(), sizeof(PairDesc), r->pairs.size(), f) == r->pairs.size();
    if (ok && h.n_pairs) ok = fread(r->counts.data(), sizeof(int32_t), r->counts.size(), f) == r->counts.size();
    int64_t total = 0;
    for (size_t k = 0; ok && k < r->pairs.size(); ++k) {
        if (r->counts[k] < 0) { ok = false; break; }
        r->offsets[k] = (uint64_t)total;      // segment 0
        total += r->counts[k];
    }
    if (ok && total != h.n_matches) ok = false;
    if (ok) {
        esfm_results::Segment sg{nullptr, (size_t)total, nullptr};
        if (total > 0) {
            sg.ptr = (esfm_dmatch_t*)malloc((size_t)total * sizeof(esfm_dmatch_t));
            ok = sg.ptr && fread(sg.ptr, sizeof(esfm_dmatch_t), (size_t)total, f) == (size_t)total;
        }
        r->segments.push_back(sg);
        r->total_matches = total;
    }
    fclose(f);
    if (!ok) {
        esfm_results_destroy(r);
        return fail(ESFM_ERR_INVALID, "esfm_results_load: %s is truncated or inconsistent", path);
    }
    *out = r;
    return ESFM_OK;
}
