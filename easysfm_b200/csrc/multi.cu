// multi.cu -- esfm_multi_*: the all-pairs job on several GPUs of one box, driven by ONE host process.
//
// The reference's caller is a single-threaded pair loop in one process (cpp_code/test/sfm.cpp:32,140-161), so the drop-in
// keeps that shape: one call uploads the bank to device 0, replicates it with one ncclBroadcast over NVLink / NVSwitch,
// deals the N(N-1)/2 independent image pairs to the devices and merges every device's compacted matches into one results
// object in the caller's pair order.  There is no inter-GPU traffic while matching (SURVEY 8e: the path shards by pairs);
// each device returns its matches over its own PCIe link, chunk by chunk, overlapped with its next chunk's sweep
// (match_pairs_impl in capi.cu).  "Gather to rank 0" is therefore N concurrent device->host streams into one process.
//
// NCCL is loaded at run time (dlopen) so that the single-GPU library has no link-time dependency on it.
#include <dlfcn.h>

#include <algorithm>
#include <chrono>
#include <cstdlib>
#include <cstring>
#include <new>
#include <numeric>

#include "host_internal.h"

using namespace esfm;

namespace {

// The five NCCL entry points used, with the types of nccl.h (2.x ABI: ncclUint8 == 1, ncclSuccess == 0).
typedef struct ncclComm* ncclComm_t;
typedef int ncclResult_t;
constexpr int kNcclUint8 = 1;
struct NcclApi {
    void* lib = nullptr;
    ncclResult_t (*CommInitAll)(ncclComm_t*, int, const int*) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    ncclResult_t (*Broadcast)(const void*, void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
};

int load_nccl(NcclApi& api) {
    const char* names[] = {getenv("ESFM_NCCL_LIBRARY"), "libnccl.so.2", "libnccl.so"};
    for (const char* n : names) {
        if (!n || !*n) continue;
        api.lib = dlopen(n, RTLD_NOW | RTLD_LOCAL);
        if (api.lib) break;
    }
    if (!api.lib) return fail(ESFM_ERR_CUDA, "esfm_multi_init: cannot load NCCL (libnccl.so.2; set ESFM_NCCL_LIBRARY): %s", dlerror());
    api.CommInitAll = (decltype(api.CommInitAll))dlsym(api.lib, "ncclCommInitAll");
    api.CommDestroy = (decltype(api.CommDestroy))dlsym(api.lib, "ncclCommDestroy");
    api.GroupStart = (decltype(api.GroupStart))dlsym(api.lib, "ncclGroupStart");
    api.GroupEnd = (decltype(api.GroupEnd))dlsym(api.lib, "ncclGroupEnd");
    api.Broadcast = (decltype(api.Broadcast))dlsym(api.lib, "ncclBroadcast");
    api.GetErrorString = (decltype(api.GetErrorString))dlsym(api.lib, "ncclGetErrorString");
    if (!api.CommInitAll || !api.CommDestroy || !api.GroupStart || !api.GroupEnd || !api.Broadcast || !api.GetErrorString)
        return fail(ESFM_ERR_CUDA, "esfm_multi_init: the NCCL library lacks a required symbol");
    return ESFM_OK;
}

double now_ms() {
    return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

// The calling thread's current CUDA device is left as it was found (the process may use torch / its own CUDA code on it).
struct DeviceRestore {
    int dev = -1;
    DeviceRestore() { if (cudaGetDevice(&dev) != cudaSuccess) { cudaGetLastError(); dev = -1; } }
    ~DeviceRestore() { if (dev >= 0) cudaSetDevice(dev); }
};

constexpr int kDealBlock = 64;     // consecutive pairs dealt together (they share the query frame: L2 locality inside a device);
                                   // small batches use smaller blocks so that every device still gets ~8 of them

}  // namespace

struct esfm_multi {
    int n = 0;
    std::vector<int> devices;
    std::vector<esfm_ctx*> ctx;
    bool distinct = true;          // every device listed once (NCCL needs that); otherwise replicas are filled by device copies
    NcclApi nccl;
    std::vector<ncclComm_t> comms;
    esfm_multi_timing_t timing{};
};

struct esfm_multi_bank {
    esfm_multi* m = nullptr;
    std::vector<esfm_bank*> bank;  // bank[0] is the primary (host-fed) replica
    bool committed = false;
};

extern "C" int esfm_multi_destroy(esfm_multi_t* m) {
    if (!m) return ESFM_OK;
    for (ncclComm_t c : m->comms)
        if (c && m->nccl.CommDestroy) m->nccl.CommDestroy(c);
    for (esfm_ctx* c : m->ctx) esfm_destroy(c);
    // (the NCCL library stays loaded: dlclose of a CUDA-using library at exit is not worth the risk)
    delete m;
    return ESFM_OK;
}

extern "C" int esfm_multi_init(int n_devices, const int* device_ids, esfm_multi_t** out) {
    if (!out) return fail(ESFM_ERR_INVALID, "esfm_multi_init: multi is NULL");
    *out = nullptr;
    if (n_devices < 1 || n_devices > 64) return fail(ESFM_ERR_INVALID, "esfm_multi_init: n_devices %d out of range [1,64]", n_devices);
    DeviceRestore restore;
    esfm_multi* m = new (std::nothrow) esfm_multi();
    if (!m) return fail(ESFM_ERR_NOMEM, "out of host memory");
    m->n = n_devices;
    for (int k = 0; k < n_devices; ++k) m->devices.push_back(device_ids ? device_ids[k] : k);
    std::vector<int> sorted = m->devices;
    std::sort(sorted.begin(), sorted.end());
    m->distinct = std::adjacent_find(sorted.begin(), sorted.end()) == sorted.end();
    for (int k = 0; k < n_devices; ++k) {
        esfm_ctx* c = nullptr;
        if (int rc = esfm_init(m->devices[(size_t)k], nullptr, &c)) { esfm_multi_destroy(m); return rc; }
        m->ctx.push_back(c);
        // a multi-device job streams every device's matches through a few pinned slots: allocate them here, not on the job's clock
        if (int rc = reserve_stream_slots(c)) { esfm_multi_destroy(m); return rc; }
    }
    if (n_devices > 1 && m->distinct) {
        if (int rc = load_nccl(m->nccl)) { esfm_multi_destroy(m); return rc; }
        m->comms.assign((size_t)n_devices, nullptr);
        const ncclResult_t r = m->nccl.CommInitAll(m->comms.data(), n_devices, m->devices.data());
        if (r != 0) {
            const int rc = fail(ESFM_ERR_CUDA, "ncclCommInitAll failed: %s", m->nccl.GetErrorString(r));
            m->comms.clear();
            esfm_multi_destroy(m);
            return rc;
        }
        // NCCL connects its channels lazily at the first collective (hundreds of ms): do that here with a 16-byte broadcast
        ncclResult_t w = m->nccl.GroupStart();
        for (int k = 0; k < n_devices && w == 0; ++k) {
            cudaSetDevice(m->devices[(size_t)k]);
            void* buf = m->ctx[(size_t)k]->buf[1].d_cursor;
            w = m->nccl.Broadcast(buf, buf, 16, kNcclUint8, 0, m->comms[(size_t)k], m->ctx[(size_t)k]->stream);
        }
        const ncclResult_t w2 = m->nccl.GroupEnd();
        for (int k = 0; k < n_devices; ++k) {
            cudaSetDevice(m->devices[(size_t)k]);
            cudaStreamSynchronize(m->ctx[(size_t)k]->stream);
        }
        if (w != 0 || w2 != 0) {
            const int rc = fail(ESFM_ERR_CUDA, "NCCL warm-up broadcast failed: %s", m->nccl.GetErrorString(w != 0 ? w : w2));
            esfm_multi_destroy(m);
            return rc;
        }
    }
    *out = m;
    return ESFM_OK;
}

extern "C" int esfm_multi_device_count(esfm_multi_t* m, int* n) {
    if (!m || !n) return fail(ESFM_ERR_INVALID, "esfm_multi_device_count: NULL argument");
    *n = m->n;
    return ESFM_OK;
}

extern "C" int esfm_multi_ctx(esfm_multi_t* m, int k, esfm_ctx_t** ctx) {
    if (!m || !ctx) return fail(ESFM_ERR_INVALID, "esfm_multi_ctx: NULL argument");
    if (k < 0 || k >= m->n) return fail(ESFM_ERR_INVALID, "device slot %d out of range [0,%d)", k, m->n);
    *ctx = m->ctx[(size_t)k];
    return ESFM_OK;
}

extern "C" int esfm_multi_timing(esfm_multi_t* m, esfm_multi_timing_t* out) {
    if (!m || !out) return fail(ESFM_ERR_INVALID, "esfm_multi_timing: NULL argument");
    *out = m->timing;
    return ESFM_OK;
}

// ------------------------------------------------------------------------------------------------
// bank: fed on device 0, replicated with one broadcast
// ------------------------------------------------------------------------------------------------
extern "C" int esfm_multi_bank_destroy(esfm_multi_bank_t* mb) {
    if (!mb) return ESFM_OK;
    for (esfm_bank* b : mb->bank) esfm_bank_destroy(b);
    delete mb;
    return ESFM_OK;
}

extern "C" int esfm_multi_bank_create(esfm_multi_t* m, esfm_kind kind, int n_frames, esfm_multi_bank_t** out) {
    if (!m || !out) return fail(ESFM_ERR_INVALID, "esfm_multi_bank_create: NULL argument");
    *out = nullptr;
    esfm_multi_bank* mb = new (std::nothrow) esfm_multi_bank();
    if (!mb) return fail(ESFM_ERR_NOMEM, "out of host memory");
    mb->m = m;
    for (int k = 0; k < m->n; ++k) {
        esfm_bank* b = nullptr;
        if (int rc = esfm_bank_create(m->ctx[(size_t)k], kind, n_frames, &b)) { esfm_multi_bank_destroy(mb); return rc; }
        mb->bank.push_back(b);
    }
    *out = mb;
    return ESFM_OK;
}

extern "C" int esfm_multi_bank_set_frame(esfm_multi_bank_t* mb, int frame_id, const void* data, int rows, int cols, size_t step_bytes) {
    if (!mb) return fail(ESFM_ERR_INVALID, "bank is NULL");
    if (mb->committed) return fail(ESFM_ERR_STATE, "esfm_multi_bank_set_frame: bank already committed");
    return esfm_bank_set_frame(mb->bank[0], frame_id, data, rows, cols, step_bytes);
}

extern "C" int esfm_multi_bank_primary(esfm_multi_bank_t* mb, esfm_bank_t** primary) {
    if (!mb || !primary) return fail(ESFM_ERR_INVALID, "esfm_multi_bank_primary: NULL argument");
    *primary = mb->bank[0];
    return ESFM_OK;
}

extern "C" int esfm_multi_bank_commit(esfm_multi_bank_t* mb) {
    if (!mb) return fail(ESFM_ERR_INVALID, "bank is NULL");
    if (mb->committed) return fail(ESFM_ERR_STATE, "bank already committed");
    esfm_multi* m = mb->m;
    DeviceRestore restore;
    const double t0 = now_ms();
    esfm_bank* p = mb->bank[0];
    // device 0: host frames (esfm_bank_set_frame / _pinned) or rows written on the device (esfm_bank_alloc_device)
    if (!p->committed) {
        if (int rc = p->device_allocated ? esfm_bank_commit_device(p) : esfm_bank_commit(p)) return rc;
    }
    const double t1 = now_ms();
    m->timing.used_nccl = 0;
    if (m->n > 1) {
        for (int k = 1; k < m->n; ++k) {
            esfm_bank* r = mb->bank[(size_t)k];
            for (int f = 0; f < p->n_frames; ++f)
                if (int rc = esfm_bank_set_frame_rows(r, f, p->rows[(size_t)f])) return rc;
            if (int rc = esfm_bank_alloc_device(r)) return rc;
        }
        const size_t bytes = (size_t)p->row_off[(size_t)p->n_frames] * p->row_bytes();
        if (bytes > 0) {
            if (m->distinct) {
                // ONE broadcast of the raw row-major bank, device 0 -> every other device, straight into the replicas' buffers
                ncclResult_t r = m->nccl.GroupStart();
                for (int k = 0; k < m->n && r == 0; ++k) {
                    CUDA_TRY(cudaSetDevice(m->devices[(size_t)k]));
                    r = m->nccl.Broadcast(p->d_rows, mb->bank[(size_t)k]->d_rows, bytes, kNcclUint8, 0, m->comms[(size_t)k], m->ctx[(size_t)k]->stream);
                }
                const ncclResult_t r2 = m->nccl.GroupEnd();
                if (r != 0 || r2 != 0) return fail(ESFM_ERR_CUDA, "ncclBroadcast of the descriptor bank failed: %s", m->nccl.GetErrorString(r != 0 ? r : r2));
                m->timing.used_nccl = 1;
            } else {
                for (int k = 1; k < m->n; ++k) {
                    CUDA_TRY(cudaSetDevice(m->devices[(size_t)k]));
                    CUDA_TRY(cudaMemcpyPeerAsync(mb->bank[(size_t)k]->d_rows, m->devices[(size_t)k], p->d_rows, m->devices[0], bytes, m->ctx[(size_t)k]->stream));
                }
            }
            for (int k = 0; k < m->n; ++k) {
                CUDA_TRY(cudaSetDevice(m->devices[(size_t)k]));
                CUDA_TRY(cudaStreamSynchronize(m->ctx[(size_t)k]->stream));
            }
        }
        for (int k = 1; k < m->n; ++k)
            if (int rc = esfm_bank_commit_device(mb->bank[(size_t)k])) return rc;
    }
    const double t2 = now_ms();
    m->timing.broadcast_ms = t2 - t1;
    m->timing.commit_ms = t2 - t0;
    mb->committed = true;
    return ESFM_OK;
}

// ------------------------------------------------------------------------------------------------
// matching: deal pairs by work, one worker thread per device, merge
// ------------------------------------------------------------------------------------------------
extern "C" int esfm_multi_match_pairs(esfm_multi_bank_t* mb, const esfm_pair_t* pairs, int64_t n_pairs, double ratio, int cross_check,
                                      int keep, esfm_results_t** out) {
    if (!mb || !out) return fail(ESFM_ERR_INVALID, "esfm_multi_match_pairs: NULL argument");
    *out = nullptr;
    if (!mb->committed) return fail(ESFM_ERR_STATE, "esfm_multi_match_pairs: bank not committed");
    if (n_pairs < 0 || (n_pairs > 0 && !pairs)) return fail(ESFM_ERR_INVALID, "esfm_multi_match_pairs: bad pair list");
    esfm_multi* m = mb->m;
    const esfm_bank* p = mb->bank[0];
    const int nd = m->n;
    for (int64_t k = 0; k < n_pairs; ++k)
        if (pairs[k].query < 0 || pairs[k].query >= p->n_frames || pairs[k].train < 0 || pairs[k].train >= p->n_frames)
            return fail(ESFM_ERR_INVALID, "pair %lld = (%d,%d) out of range [0,%d)", (long long)k, pairs[k].query, pairs[k].train, p->n_frames);
    DeviceRestore restore;
    const double t0 = now_ms();

    // Deal blocks of consecutive pairs to the least-loaded device, work = rows_q * rows_t (SURVEY 8e: ragged frames would
    // unbalance a deal by count).  Deterministic; every device keeps its pairs in the caller's order.
    std::vector<std::vector<int64_t>> mine((size_t)nd);
    std::vector<double> load((size_t)nd, 0.0);
    const int64_t block = std::max<int64_t>(1, std::min<int64_t>(kDealBlock, n_pairs / ((int64_t)nd * 8)));
    for (int64_t b0 = 0; b0 < n_pairs; b0 += block) {
        const int64_t b1 = std::min<int64_t>(n_pairs, b0 + block);
        double w = 0.0;
        for (int64_t k = b0; k < b1; ++k) w += (double)p->rows[(size_t)pairs[k].query] * (double)p->rows[(size_t)pairs[k].train] + 1.0;
        const int d = (int)(std::min_element(load.begin(), load.end()) - load.begin());
        load[(size_t)d] += w;
        for (int64_t k = b0; k < b1; ++k) mine[(size_t)d].push_back(k);
    }
    const double mean = std::accumulate(load.begin(), load.end(), 0.0) / nd;
    m->timing.work_imbalance = mean > 0 ? *std::max_element(load.begin(), load.end()) / mean - 1.0 : 0.0;

    std::vector<esfm_results*> part((size_t)nd, nullptr);
    std::vector<int> rcs((size_t)nd, ESFM_OK);
    std::vector<std::string> errs((size_t)nd);
    std::vector<double> dev_ms((size_t)nd, 0.0);
    auto work = [&](int d) {
        const double s0 = now_ms();
        std::vector<esfm_pair_t> list(mine[(size_t)d].size());
        for (size_t i = 0; i < list.size(); ++i) list[i] = pairs[mine[(size_t)d][i]];
        rcs[(size_t)d] = match_pairs_impl(mb->bank[(size_t)d], list.data(), (int64_t)list.size(), ratio, cross_check, MatchOpts{true, keep}, &part[(size_t)d]);
        if (rcs[(size_t)d]) errs[(size_t)d] = g_last_error;      // (the message lives in the worker's thread-local slot)
        dev_ms[(size_t)d] = now_ms() - s0;
    };
    if (nd == 1) {
        work(0);
    } else {
        std::vector<std::thread> threads;
        for (int d = 0; d < nd; ++d) threads.emplace_back(work, d);
        for (auto& t : threads) t.join();
    }
    for (int d = 0; d < nd; ++d) {
        if (rcs[(size_t)d]) {
            const int rc = fail(rcs[(size_t)d], "device slot %d (cuda:%d): %s", d, m->devices[(size_t)d], errs[(size_t)d].c_str());
            for (esfm_results* r : part) esfm_results_destroy(r);
            return rc;
        }
    }

    // merge: one results object in the caller's pair order; the devices' match segments are adopted, not copied
    esfm_results* res = new (std::nothrow) esfm_results();
    if (!res) { for (esfm_results* r : part) esfm_results_destroy(r); return fail(ESFM_ERR_NOMEM, "out of host memory"); }
    res->ctx = nullptr;
    res->kind = p->kind;
    res->ratio = ratio;
    res->cross_check = cross_check ? 1 : 0;
    res->keep = keep;
    res->frame_rows.assign(p->rows.begin(), p->rows.end());
    res->fetched = true;
    res->pairs.resize((size_t)n_pairs);
    res->counts.assign((size_t)n_pairs, 0);
    res->offsets.assign((size_t)n_pairs, 0);
    if (keep == ESFM_KEEP_DIGESTS) res->digests.assign((size_t)n_pairs, 0);
    for (int64_t k = 0; k < n_pairs; ++k) {
        res->pairs[(size_t)k].q_frame = pairs[k].query;
        res->pairs[(size_t)k].t_frame = pairs[k].train;
    }
    for (int d = 0; d < nd; ++d) {
        esfm_results* r = part[(size_t)d];
        const uint64_t seg_base = (uint64_t)res->segments.size();
        for (auto& s : r->segments) res->segments.push_back(s);
        r->segments.clear();                       // ownership moved
        const auto& ids = mine[(size_t)d];
        for (size_t i = 0; i < ids.size(); ++i) {
            const size_t g = (size_t)ids[i];
            res->counts[g] = r->counts[i];
            const uint64_t o = r->offsets[i];
            res->offsets[g] = (((o >> 40) + seg_base) << 40) | (o & (((uint64_t)1 << 40) - 1));
            if (keep == ESFM_KEEP_DIGESTS) res->digests[g] = r->digests[i];
        }
        res->total_matches += r->total_matches;
        esfm_results_destroy(r);
    }
    m->timing.match_ms = now_ms() - t0;
    m->timing.device_ms_max = *std::max_element(dev_ms.begin(), dev_ms.end());
    m->timing.device_ms_min = *std::min_element(dev_ms.begin(), dev_ms.end());
    *out = res;
    return ESFM_OK;
}

extern "C" int esfm_multi_match_all_pairs(esfm_multi_bank_t* mb, double ratio, int cross_check, int keep, esfm_results_t** out) {
    if (!mb || !out) return fail(ESFM_ERR_INVALID, "esfm_multi_match_all_pairs: NULL argument");
    std::vector<esfm_pair_t> pairs;
    const int n = mb->bank[0]->n_frames;
    pairs.reserve((size_t)n * (size_t)(n > 0 ? n - 1 : 0) / 2);
    for (int i = 0; i < n; ++i)           // cpp_code/test/sfm.cpp:140
        for (int j = 0; j < i; ++j) {     // cpp_code/test/sfm.cpp:143
            esfm_pair_t pr;
            pr.query = i;
            pr.train = j;
            pairs.push_back(pr);
        }
    return esfm_multi_match_pairs(mb, pairs.data(), (int64_t)pairs.size(), ratio, cross_check, keep, out);
}

// ------------------------------------------------------------------------------------------------
// verification of a results batch: deal pairs by match count, one worker thread per device, merge
// ------------------------------------------------------------------------------------------------
extern "C" int esfm_multi_two_view_results(esfm_multi_t* m, esfm_results_t* matches, int n_frames, const int64_t* kp_off, const float* kp_xy,
                                           const double* K, int k_per_frame, const esfm_two_view_params_t* params, int min_pair_matches,
                                           esfm_results_t** inliers, esfm_two_view_t* out) {
    TvJob job;
    if (int rc = two_view_job("esfm_multi_two_view_results", matches, n_frames, kp_off, kp_xy, K, k_per_frame, params, min_pair_matches, inliers, out, &job))
        return rc;
    if (!m) return fail(ESFM_ERR_INVALID, "esfm_multi_two_view_results: NULL argument");
    DeviceRestore restore;
    const double t0 = now_ms();
    const int nd = m->n;
    const int64_t n_pairs = (int64_t)matches->pairs.size();
    // blocks of consecutive pairs to the least-loaded device, work = matches + 1 (the RANSAC of a pair scores every match)
    std::vector<TvShare> shares((size_t)nd);
    std::vector<double> load((size_t)nd, 0.0);
    const int64_t block = std::max<int64_t>(1, std::min<int64_t>(kDealBlock, n_pairs / ((int64_t)nd * 8)));
    for (int64_t b0 = 0; b0 < n_pairs; b0 += block) {
        const int64_t b1 = std::min<int64_t>(n_pairs, b0 + block);
        double w = 0.0;
        for (int64_t k = b0; k < b1; ++k) w += (double)matches->counts[(size_t)k] + 1.0;
        const int d = (int)(std::min_element(load.begin(), load.end()) - load.begin());
        load[(size_t)d] += w;
        for (int64_t k = b0; k < b1; ++k) shares[(size_t)d].ids.push_back(k);
    }
    const double mean = std::accumulate(load.begin(), load.end(), 0.0) / nd;
    m->timing.work_imbalance = mean > 0 ? *std::max_element(load.begin(), load.end()) / mean - 1.0 : 0.0;
    std::vector<int> rcs((size_t)nd, ESFM_OK);
    std::vector<std::string> errs((size_t)nd);
    std::vector<double> dev_ms((size_t)nd, 0.0);
    auto work = [&](int d) {
        const double s0 = now_ms();
        rcs[(size_t)d] = two_view_share(m->ctx[(size_t)d], job, shares[(size_t)d]);
        if (rcs[(size_t)d]) errs[(size_t)d] = g_last_error;      // (the message lives in the worker's thread-local slot)
        dev_ms[(size_t)d] = now_ms() - s0;
    };
    if (nd == 1) {
        work(0);
    } else {
        std::vector<std::thread> threads;
        for (int d = 0; d < nd; ++d) threads.emplace_back(work, d);
        for (auto& t : threads) t.join();
    }
    // the first offending pair of the batch, else the first failing device
    int failed = -1;
    for (int d = 0; d < nd; ++d) {
        if (!rcs[(size_t)d]) continue;
        const int64_t b = shares[(size_t)d].bad_pair, fb = failed < 0 ? -1 : shares[(size_t)failed].bad_pair;
        if (failed < 0 || (b >= 0 && (fb < 0 || b < fb))) failed = d;
    }
    if (failed >= 0) return fail(rcs[(size_t)failed], "device slot %d (cuda:%d): %s", failed, m->devices[(size_t)failed], errs[(size_t)failed].c_str());
    const int rc = two_view_assemble(job, shares, inliers, out);
    m->timing.match_ms = now_ms() - t0;
    m->timing.device_ms_max = *std::max_element(dev_ms.begin(), dev_ms.end());
    m->timing.device_ms_min = *std::min_element(dev_ms.begin(), dev_ms.end());
    return rc;
}
