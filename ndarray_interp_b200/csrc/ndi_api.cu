// ndi_api.cu -- the C ABI (include/ndi_b200.h): handles, table upload, dtype dispatch and the
// host-buffer pipeline around the kernels.  No interpolation arithmetic happens on the host.
//
// Host entry points (no _dev suffix):
//   results <= 256 KB : the latency path of interp_scalar / interp / interp_into: queries and rows live in the
//                   thread's pinned workspace, which the kernel reads and writes directly; completion is a flag
//                   in that workspace (profiles/r01/latency.md).
//   larger batches : chunk by chunk, (1) the queries go up on a copy-in stream a few chunks ahead, (2) the
//                   K7 pre-pass over each chunk finds the first query the reference would fail on, (3) only
//                   the rows before it are evaluated, alternating between two streams so the D2H copy of
//                   one chunk overlaps the kernel of the next.  Rows at and after the failing query stay
//                   untouched, like the reference (interp1d/mod.rs:321,336-340).  Page-locked output arrays
//                   receive the chunks directly; ordinary pageable ones through three pinned staging
//                   buffers and a pool of copy threads.
// All per-call state lives in a thread-local workspace, so one handle can be used from many
// threads at once (the reference's &self methods are called from rayon workers).
#include <atomic>
#include <condition_variable>
#include <deque>
#include <functional>
#include <thread>
#include <unordered_map>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <vector>

#include "../../include/ndi_b200.h"
#include "ndi_internal.h"

namespace ndi {

// ---- errors ----------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";
static ndi_status fail(ndi_status st, const char* fmt, ...) {
    va_list ap; va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return st;
}
static ndi_status cuda_fail(cudaError_t e, const char* what) {
    snprintf(g_err, sizeof(g_err), "%s: %s (%s)", what, cudaGetErrorString(e), cudaGetErrorName(e));
    cudaGetLastError();   // clear the sticky-free error state
    return NDI_CUDA_ERROR + (ndi_status)e;
}
#define CK(call)                                                   \
    do {                                                           \
        cudaError_t e__ = (call);                                  \
        if (e__ != cudaSuccess) return cuda_fail(e__, #call);      \
    } while (0)

// ---- device info / launch counter -------------------------------------------------------------------
static std::atomic<uint64_t> g_launches{0};
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }

const DeviceInfo& device_info() {
    static std::mutex mu;
    static std::map<int, DeviceInfo> cache;
    int dev = 0;
    cudaGetDevice(&dev);
    std::lock_guard<std::mutex> lk(mu);
    auto it = cache.find(dev);
    if (it != cache.end()) return it->second;
    DeviceInfo di{dev, 148, 48 * 1024, (size_t)126 << 20};
    int v = 0;
    if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && v > 0) di.sm_count = v;
    if (cudaDeviceGetAttribute(&v, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev) == cudaSuccess && v > 0) di.smem_optin = (size_t)v;
    if (cudaDeviceGetAttribute(&v, cudaDevAttrL2CacheSize, dev) == cudaSuccess && v > 0) di.l2_bytes = (size_t)v;
    // per-launch scratch (query binning) comes from the stream-ordered pool; keep freed blocks cached
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
        uint64_t keep = ~0ull;
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
    }
    cudaGetLastError();
    return cache.emplace(dev, di).first->second;
}

struct DeviceGuard {
    int prev = -1; bool changed = false;
    explicit DeviceGuard(int dev) {
        if (cudaGetDevice(&prev) == cudaSuccess && prev != dev) changed = cudaSetDevice(dev) == cudaSuccess;
    }
    ~DeviceGuard() { if (changed) cudaSetDevice(prev); }
};

static size_t elem_size(ndi_dtype d) { return (d == NDI_F64 || d == NDI_I64 || d == NDI_U64) ? 8 : 4; }
static bool dtype_ok(ndi_dtype d) { return d >= NDI_F32 && d <= NDI_U64; }

template <class F>
static ndi_status dispatch(ndi_dtype d, F&& f) {
    switch (d) {
    case NDI_F32: return f(float{});
    case NDI_F64: return f(double{});
    case NDI_I32: return f(int32_t{});
    case NDI_I64: return f(int64_t{});
    case NDI_U32: return f(uint32_t{});
    case NDI_U64: return f(uint64_t{});
    default: return fail(NDI_UNSUPPORTED_DTYPE, "unsupported dtype %d", (int)d);
    }
}
template <class F>
static ndi_status dispatch_float(ndi_dtype d, F&& f) {
    switch (d) {
    case NDI_F32: return f(float{});
    case NDI_F64: return f(double{});
    default: return fail(NDI_UNSUPPORTED_DTYPE, "cubic splines need a float dtype (SplineNum), got %d", (int)d);
    }
}

// ---- thread-local workspace --------------------------------------------------------------------------
constexpr size_t kChunkBytes = 64ull << 20;    // output bytes per pipeline chunk
// results up to this size (and so queries, never more bytes than their rows) go through the pinned workspace,
// which the kernel reads and writes directly
constexpr size_t kTinyBytes = 256ull << 10;

struct Workspace {
    bool ready = false;
    cudaStream_t s[2] = {nullptr, nullptr};
    cudaStream_t s_in = nullptr;              // copy-in stream of the streaming host pipeline (queries up + pre-pass, a few chunks ahead)
    cudaEvent_t feed_ev[3] = {nullptr, nullptr, nullptr};
    cudaEvent_t ev = nullptr;
    void* d_q[2] = {nullptr, nullptr}; size_t d_q_cap[2] = {0, 0};
    void* d_out[2] = {nullptr, nullptr}; size_t d_out_cap[2] = {0, 0};
    void* d_build = nullptr; size_t d_build_cap = 0;       // spline-build scratch, kept between builds (up to kBuildKeepBytes)
    unsigned long long* d_err = nullptr;      // 8 words: [0] call, [1] tiny-batch path, [4..6] chunks of the streaming pipeline
    int32_t* d_res = nullptr;                 // 2 words (grid classify result)
    uint32_t* d_scr = nullptr;                // grid classify scratch
    unsigned char* h_pin = nullptr; size_t h_pin_cap = 0;   // pinned: [err word, flag | tiny outputs | tiny queries x 2]
    unsigned char* h_stage[3] = {nullptr, nullptr, nullptr};   // pinned staging for pageable outputs (lazy)
    cudaEvent_t stage_ev[3] = {nullptr, nullptr, nullptr};
    unsigned long long seq = 0;               // completion counter of the tiny-batch path
    bool err_armed = false;                   // d_err[1] holds ~0 (re-armed by publish_kernel)
};

static Workspace* workspace(int dev, ndi_status* st) {
    static thread_local std::map<int, Workspace> per_dev;
    Workspace& w = per_dev[dev];
    *st = NDI_OK;
    if (w.ready) return &w;
    cudaError_t e;
    for (int i = 0; i < 2; ++i)
        if ((e = cudaStreamCreateWithFlags(&w.s[i], cudaStreamNonBlocking)) != cudaSuccess) { *st = cuda_fail(e, "cudaStreamCreate"); return nullptr; }
    if ((e = cudaStreamCreateWithFlags(&w.s_in, cudaStreamNonBlocking)) != cudaSuccess) { *st = cuda_fail(e, "cudaStreamCreate"); return nullptr; }
    if ((e = cudaEventCreateWithFlags(&w.ev, cudaEventDisableTiming)) != cudaSuccess) { *st = cuda_fail(e, "cudaEventCreate"); return nullptr; }
    for (int i = 0; i < 3; ++i)
        if ((e = cudaEventCreateWithFlags(&w.feed_ev[i], cudaEventDisableTiming)) != cudaSuccess) { *st = cuda_fail(e, "cudaEventCreate"); return nullptr; }
    if ((e = cudaMalloc(&w.d_err, 8 * sizeof(unsigned long long))) != cudaSuccess) { *st = cuda_fail(e, "cudaMalloc"); return nullptr; }
    if ((e = cudaMalloc(&w.d_res, 2 * sizeof(int32_t))) != cudaSuccess) { *st = cuda_fail(e, "cudaMalloc"); return nullptr; }
    if ((e = cudaMalloc(&w.d_scr, grid_classify_scratch_words() * sizeof(uint32_t))) != cudaSuccess) { *st = cuda_fail(e, "cudaMalloc"); return nullptr; }
    w.h_pin_cap = 64 + 3 * kTinyBytes;
    if ((e = cudaMallocHost(&w.h_pin, w.h_pin_cap)) != cudaSuccess) { *st = cuda_fail(e, "cudaMallocHost"); return nullptr; }
    w.ready = true;
    return &w;
}
static ndi_status grow(void** p, size_t* cap, size_t need) {
    if (*cap >= need) return NDI_OK;
    if (*p) { cudaFree(*p); *p = nullptr; *cap = 0; }
    size_t want = need + need / 4;
    cudaError_t e = cudaMalloc(p, want);
    if (e != cudaSuccess) { want = need; e = cudaMalloc(p, want); }
    if (e != cudaSuccess) return cuda_fail(e, "cudaMalloc(workspace)");
    *cap = want;
    return NDI_OK;
}

// ---- host-side copy pool -------------------------------------------------------------------------------
// Results for ordinary (pageable) host arrays are copied device -> pinned staging -> caller memory; the
// second hop is a plain memcpy, which one core cannot do at PCIe speed, so a few worker threads share it.
// One pool per process, created on first use and never destroyed (workers block on a condition variable).
constexpr size_t kStageBytes = 16ull << 20;
class CopyPool {
public:
    static CopyPool& get() { static CopyPool* p = new CopyPool(); return *p; }
    // copy asynchronously; returns a ticket for wait()
    uint64_t submit(void* dst, const void* src, size_t bytes) {
        std::unique_lock<std::mutex> lk(mu_);
        const uint64_t t = ++last_ticket_;
        const size_t parts = bytes >= (1u << 20) ? nthreads_ : 1;
        const size_t slice = ((bytes + parts - 1) / parts + 63) & ~(size_t)63;
        int n = 0;
        for (size_t off = 0; off < bytes; off += slice, ++n)
            tasks_.push_back(Task{(unsigned char*)dst + off, (const unsigned char*)src + off, bytes - off < slice ? bytes - off : slice, t});
        if (n == 0) return 0;
        pending_[t] = n;
        lk.unlock();
        work_.notify_all();
        return t;
    }
    void wait(uint64_t ticket) {
        if (!ticket) return;
        std::unique_lock<std::mutex> lk(mu_);
        done_.wait(lk, [&] { return pending_.find(ticket) == pending_.end(); });
    }
private:
    struct Task { unsigned char* dst; const unsigned char* src; size_t bytes; uint64_t ticket; };
    CopyPool() {
        unsigned hw = std::thread::hardware_concurrency();
        nthreads_ = hw >= 16 ? 8 : (hw >= 4 ? hw / 2 : 1);
        if (const char* e = getenv("NDI_COPY_THREADS")) { long v = strtol(e, nullptr, 10); if (v >= 1 && v <= 64) nthreads_ = (size_t)v; }
        for (size_t i = 0; i < nthreads_; ++i) std::thread([this] { run(); }).detach();
    }
    void run() {
        for (;;) {
            Task t;
            {
                std::unique_lock<std::mutex> lk(mu_);
                work_.wait(lk, [&] { return !tasks_.empty(); });
                t = tasks_.front(); tasks_.pop_front();
            }
            memcpy(t.dst, t.src, t.bytes);
            {
                std::lock_guard<std::mutex> lk(mu_);
                auto it = pending_.find(t.ticket);
                if (it != pending_.end() && --it->second == 0) { pending_.erase(it); done_.notify_all(); }
            }
        }
    }
    std::mutex mu_; std::condition_variable work_, done_;
    std::deque<Task> tasks_; std::unordered_map<uint64_t, int> pending_;
    uint64_t last_ticket_ = 0; size_t nthreads_ = 1;
};

static bool is_pageable_host(const void* p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return true; }
    return a.type == cudaMemoryTypeUnregistered;
}

// ---- search configuration ----------------------------------------------------------------------------
// A grid that does not fit the shared-memory budget gets a coarse table grid[0], grid[S], ... built
// once per handle; the kernels bisect the coarse table in shared memory and finish in L1/L2.
constexpr int64_t kLutPerPoint = 8;              // buckets per grid point (rounded up to a power of two)
constexpr size_t kFullStageBytes = 48 * 1024;    // stage the whole grid up to this size
constexpr size_t kCoarseBytes = 16 * 1024;       // target size of a coarse table

struct GridMeta {
    const void* grid; int64_t n; size_t elem; int uniform_hint;
    const void* coarse; int coarse_n; int coarse_shift;
    const void* lut; int lut_n; double g0d, scale;
};

// per-grid search aids owned by a handle: coarse table (two-level bisection) and bucket table
struct GridAids {
    void* coarse = nullptr; int coarse_n = 0, coarse_shift = 0;
    void* lut = nullptr; int lut_n = 0; double g0d = 0, scale = 0;
    void release() { cudaFree(coarse); cudaFree(lut); coarse = lut = nullptr; }
    GridMeta meta(const void* grid, int64_t n, size_t elem, int hint) const {
        return GridMeta{grid, n, elem, hint, coarse, coarse_n, coarse_shift, lut, lut_n, g0d, scale};
    }
};

static SearchCfg make_search(const GridMeta& gm, int mode, int64_t nq, size_t other_smem) {
    SearchCfg sc{bisect_top_step(gm.n), 0, 0, 0, 0, nullptr, nullptr, 0, 0.0, 0.0, 0};
    auto use_lut = [&]() { if (gm.lut) { sc.lut = gm.lut; sc.lut_n = gm.lut_n; sc.g0d = gm.g0d; sc.scale = gm.scale; } };
    const size_t bytes = (size_t)gm.n * gm.elem;
    // the kernels' own static shared memory (barriers, per-warp record slabs: up to 16.4 KB) comes off the budget too
    constexpr size_t kStaticSmem = 17 * 1024;
    const size_t room = device_info().smem_optin > other_smem + kStaticSmem ? device_info().smem_optin - other_smem - kStaticSmem : 0;
    auto stage = [&](size_t full_limit) {
        if (bytes <= full_limit && bytes <= room) { sc.smem = 1; sc.stage_src = gm.grid; sc.stage_n = (int)gm.n; sc.coarse_shift = 0; }
        else if (gm.coarse && (size_t)gm.coarse_n * gm.elem <= room) {
            sc.smem = 1; sc.stage_src = gm.coarse; sc.stage_n = gm.coarse_n; sc.coarse_shift = gm.coarse_shift;
        }
    };
    switch (mode) {
    case NDI_SEARCH_BINARY_GLOBAL: break;
    case NDI_SEARCH_BINARY_SMEM: stage(gm.coarse ? kFullStageBytes : room); break;
    case NDI_SEARCH_UNIFORM_GUESS: sc.guess = 1; break;
    case NDI_SEARCH_BUCKET_LUT: use_lut(); break;
    case NDI_SEARCH_MERGE: sc.merge = 1; break;
    default:   // AUTO: O(1) guess on grids where it always hits, else the bucket table;
               // without either (no handle), shared-memory bisection for big batches
        // (Measured and dropped, profiles/r02/ab_eval_changes.md: staging an even grid in shared memory so that the
        // guess's two verification reads come from there -- C5a 17.007 against 17.015 ms, C4 0.5408 / 0.5403: the
        // 8 - 16 KB grids are L1-resident anyway.)
        if (gm.uniform_hint) sc.guess = 1;
        else if (gm.lut) use_lut();
        else if (nq >= 32768) stage(kFullStageBytes);
        break;
    }
    return sc;
}

// search aids of one (non-uniform) grid, built once per handle on stream st (synchronises):
//  - coarse table for a grid too large to stage whole (strided device-to-device copy)
//  - bucket table for the O(1) search
static ndi_status build_aids(ndi_dtype dtype, const void* grid, int64_t n, cudaStream_t st, GridAids* aids) {
    const size_t elem = elem_size(dtype);
    *aids = GridAids{};
    if ((size_t)n * elem > kFullStageBytes) {
        int sh = 1;
        while ((((size_t)n + ((size_t)1 << sh) - 1) >> sh) * elem > kCoarseBytes) ++sh;
        const size_t S = (size_t)1 << sh;
        const int count = (int)(((size_t)n + S - 1) / S);
        CK(cudaMalloc(&aids->coarse, (size_t)count * elem));
        CK(cudaMemcpy2DAsync(aids->coarse, elem, grid, S * elem, elem, (size_t)count, cudaMemcpyDeviceToDevice, st));
        aids->coarse_n = count; aids->coarse_shift = sh;
    }
    // bucket table: ~4 buckets per grid point
    unsigned char ends[16];
    CK(cudaMemcpyAsync(ends, grid, elem, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(ends + 8, (const unsigned char*)grid + (size_t)(n - 1) * elem, elem, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    int nb = 16;
    while (nb < kLutPerPoint * n && nb < (1 << 24)) nb <<= 1;
    while ((size_t)nb * lut_entry_bytes(elem) > ((size_t)128 << 20) && nb > 16) nb >>= 1;   // keep the table well inside L2
    double g0d, scale;
    if (dtype == NDI_F32) {
        float a, b; memcpy(&a, ends, 4); memcpy(&b, ends + 8, 4);
        const float sc = (float)nb / (b - a);            // same float arithmetic as bucket_of()
        g0d = a; scale = sc;
    } else if (dtype == NDI_F64) {
        double a, b; memcpy(&a, ends, 8); memcpy(&b, ends + 8, 8);
        g0d = a; scale = (double)nb / (b - a);
    } else if (dtype == NDI_I64) {
        int64_t a, b; memcpy(&a, ends, 8); memcpy(&b, ends + 8, 8);
        g0d = (double)a; scale = (double)nb / ((double)b - (double)a);
    } else if (dtype == NDI_U64) {
        uint64_t a, b; memcpy(&a, ends, 8); memcpy(&b, ends + 8, 8);
        g0d = (double)a; scale = (double)nb / ((double)b - (double)a);
    } else if (dtype == NDI_U32) {
        uint32_t a, b; memcpy(&a, ends, 4); memcpy(&b, ends + 8, 4);
        g0d = a; scale = (double)nb / ((double)b - (double)a);
    } else {
        int32_t a, b; memcpy(&a, ends, 4); memcpy(&b, ends + 8, 4);
        g0d = a; scale = (double)nb / ((double)b - (double)a);
    }
    if (scale > 0 && scale < 1e300 && scale == scale) {
        CK(cudaMalloc(&aids->lut, (size_t)nb * lut_entry_bytes(elem)));
        ndi_status s2 = dispatch(dtype, [&](auto tag) -> ndi_status {
            using T = decltype(tag);
            CK(launch_build_lut<T>((const T*)grid, n, g0d, scale, nb, aids->lut, st));
            return NDI_OK;
        });
        if (s2 != NDI_OK) return s2;
        aids->lut_n = nb; aids->g0d = g0d; aids->scale = scale;
    }
    CK(cudaStreamSynchronize(st));
    return NDI_OK;
}

}  // namespace ndi

using namespace ndi;

// ---- handles ---------------------------------------------------------------------------------------------
constexpr int kNotBuilt = INT32_MIN;
struct ndi_interp1d {
    ndi_dtype dtype; int device; int64_t n, w;
    void* x; void* data; void* a; void* b;
    bool owns_tables, owns_coeffs;
    int uniform_hint; int search_mode;
    int fast_tables = 0;             // f32: every data value is 0 or in [2^-56, 2^30] (hoisted-reciprocal division allowed)
    void* pair = nullptr;            // pair table for thin-row Linear (ndi_eval.cu: rows i, i+1 interleaved), owned
    int build_mode = NDI_BUILD_AUTO, build_levels = 0;   // spline solve: reference order or row-split (ndi_rowsplit.cu)
    int built_levels = kNotBuilt;    // how the current coefficients were built: 0 reference order, L > 0 row-split levels, -m partition blocks
    double nak_pivot = -1.0;         // last eliminated pivot of the NotAKnot system relative to its diagonal entry (< 0: not formed yet)
    GridAids aids;
    GridMeta meta() const { return aids.meta(x, n, elem_size(dtype), uniform_hint); }
};
struct ndi_interp2d {
    ndi_dtype dtype; int device; int64_t n, m, w;
    void* x; void* y; void* data;
    bool owns_tables;
    int hint_x, hint_y; int search_mode;
    int bin_mode = NDI_BIN_AUTO; int band_rows = 0;   // locality binning of query batches (ndi_bin.cu)
    int fast_tables = 0;
    GridAids aids_x, aids_y;
    GridMeta meta_x() const { return aids_x.meta(x, n, elem_size(dtype), hint_x); }
    GridMeta meta_y() const { return aids_y.meta(y, m, elem_size(dtype), hint_y); }
};

// upload or adopt one table
static ndi_status take_table(const void* src, size_t bytes, uint32_t flags, cudaStream_t st, void** dst, bool* owned) {
    if ((flags & NDI_DEVICE_POINTERS) && (flags & NDI_BORROW)) { *dst = const_cast<void*>(src); *owned = false; return NDI_OK; }
    CK(cudaMalloc(dst, bytes ? bytes : 1));
    *owned = true;
    if (bytes) CK(cudaMemcpyAsync(*dst, src, bytes, (flags & NDI_DEVICE_POINTERS) ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, st));
    return NDI_OK;
}

// K1 on an uploaded grid: Monotonic enum and the uniform-guess flag
static ndi_status classify_grid(ndi_dtype dtype, const void* x_dev, int64_t n, Workspace* ws, int32_t res[2]) {
    ndi_status st = dispatch(dtype, [&](auto tag) -> ndi_status {
        using T = decltype(tag);
        CK(launch_grid_classify<T>((const T*)x_dev, n, ws->d_res, ws->d_scr, ws->s[0]));
        return NDI_OK;
    });
    if (st != NDI_OK) return st;
    CK(cudaMemcpyAsync(ws->h_pin, ws->d_res, 2 * sizeof(int32_t), cudaMemcpyDeviceToHost, ws->s[0]));
    CK(cudaStreamSynchronize(ws->s[0]));
    memcpy(res, ws->h_pin, 2 * sizeof(int32_t));
    return NDI_OK;
}

// one pass over an f32 table: may the kernels use the hoisted-reciprocal division? (ndi_device.cuh)
static ndi_status scan_fast_tables(ndi_dtype dtype, const void* data_dev, size_t count, Workspace* ws, int* fast) {
    *fast = 0;
    if (dtype == NDI_F64) { *fast = 1; return NDI_OK; }   // f64 checks every quotient itself (div_ok): no scan needed
    if (dtype != NDI_F32) return NDI_OK;
    const int32_t one = 1;
    CK(cudaMemcpyAsync(ws->d_res, &one, sizeof(one), cudaMemcpyHostToDevice, ws->s[0]));
    CK(launch_table_fast_div((const float*)data_dev, count, ws->d_res, ws->s[0]));
    CK(cudaMemcpyAsync(ws->h_pin, ws->d_res, sizeof(int32_t), cudaMemcpyDeviceToHost, ws->s[0]));
    CK(cudaStreamSynchronize(ws->s[0]));
    int32_t v; memcpy(&v, ws->h_pin, sizeof(v));
    *fast = v;
    return NDI_OK;
}

// Dense device copy of a strided view (SURVEY.md section 8(f) rank 4: views and negative strides without a
// host-side copy).  `base` addresses the view's FIRST logical element; strides are in elements.  A host view
// whose memory span is at most twice its element count is uploaded as it lies and gathered on the device
// (launch_pack_strided); a sparser one is gathered by the host into a staging buffer first, because moving
// the whole span over PCIe would cost more than the gather.
static ndi_status pack_view(const void* base, size_t es, int ndim, const int64_t* shape, const int64_t* strides,
                            bool device_src, cudaStream_t st, void** dense) {
    *dense = nullptr;
    if (ndim < 1 || ndim > kMaxDims || !shape || !strides) return fail(NDI_INVALID_ARGUMENT, "views need 1..%d dimensions", kMaxDims);
    StridedDesc d; d.ndim = ndim;
    long long count = 1, lo = 0, hi = 0, dense_stride = 1;
    bool is_dense = true;
    for (int k = ndim - 1; k >= 0; --k) {
        if (shape[k] < 1) return fail(NDI_INVALID_ARGUMENT, "empty view (shape[%d] = %lld)", k, (long long)shape[k]);
        d.shape[k] = shape[k]; d.stride[k] = strides[k];
        const long long reach = (long long)(shape[k] - 1) * strides[k];
        if (reach < 0) lo += reach; else hi += reach;
        if (shape[k] > 1 && strides[k] != dense_stride) is_dense = false;
        dense_stride *= shape[k];
        count *= shape[k];
    }
    const size_t bytes = (size_t)count * es;
    CK(cudaMalloc(dense, bytes));
    auto bail = [&](ndi_status s) { cudaFree(*dense); *dense = nullptr; return s; };
#define CKP(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) return bail(cuda_fail(e_, #call)); } while (0)
    if (is_dense) {
        CKP(cudaMemcpyAsync(*dense, base, bytes, device_src ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, st));
        return NDI_OK;
    }
    const long long span = hi - lo + 1;
    const unsigned char* first = (const unsigned char*)base + lo * (long long)es;     // lowest address the view touches
    if (device_src) {
        CKP(launch_pack_strided(first, -lo, d, es, count, *dense, st));
        return NDI_OK;
    }
    if (span <= 2 * count + 4096) {
        void* raw = nullptr;
        CKP(cudaMallocAsync(&raw, (size_t)span * es, st));
        cudaError_t e = cudaMemcpyAsync(raw, first, (size_t)span * es, cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess) e = launch_pack_strided(raw, -lo, d, es, count, *dense, st);
        cudaFreeAsync(raw, st);
        if (e != cudaSuccess) return bail(cuda_fail(e, "strided upload"));
        return NDI_OK;
    }
    std::vector<unsigned char> stage(bytes);
    std::vector<long long> idx((size_t)ndim, 0);
    long long off = 0;
    for (long long i = 0; i < count; ++i) {
        memcpy(stage.data() + (size_t)i * es, (const unsigned char*)base + off * (long long)es, es);
        for (int k = ndim - 1; k >= 0; --k) {                      // odometer over the logical index
            off += strides[k];
            if (++idx[(size_t)k] < shape[k]) break;
            off -= strides[k] * shape[k]; idx[(size_t)k] = 0;
        }
    }
    CKP(cudaMemcpyAsync(*dense, stage.data(), bytes, cudaMemcpyHostToDevice, st));
    CKP(cudaStreamSynchronize(st));                                // the staging buffer goes away
#undef CKP
    return NDI_OK;
}

// Pair table for Linear on thin rows (ndi_eval.cu: interp1d_linear_pair_kernel): twice the table, so only while
// it stays comfortably L2-resident -- beyond that the gathers are DRAM sectors either way and nothing is gained.
constexpr size_t kPairMaxBytes = 48ull << 20;
static ndi_status build_pair_table(ndi_interp1d* h, cudaStream_t st) {
    const size_t es = elem_size(h->dtype);
    const size_t bytes = (size_t)(h->n - 1) * 2 * (size_t)h->w * es;
    if (!pair_table_shape_ok(h->w, es) || bytes > kPairMaxBytes || ((uintptr_t)h->data & 15)) return NDI_OK;
    CK(cudaMalloc(&h->pair, bytes));
    ndi_status s2 = dispatch(h->dtype, [&](auto tag) -> ndi_status {
        using T = decltype(tag);
        CK(launch_pack_pairs<T>((const T*)h->data, h->n, h->w, (T*)h->pair, st));
        return NDI_OK;
    });
    if (s2 != NDI_OK) return s2;
    CK(cudaStreamSynchronize(st));
    return NDI_OK;
}

// A copy of handle h on another device: fill(c, copy) points the copy c at its own device arrays, made with
// copy(&dst, src, bytes) (an NVLink peer copy), before anything in it can fail; a clone that fails is destroyed.
template <class H, class Fill>
static ndi_status clone_to_device(const H* h, int32_t device, H** out, ndi_status (*destroy)(H*), Fill&& fill) {
    if (!h || !out) return fail(NDI_INVALID_ARGUMENT, "null pointer");
    *out = nullptr;
    DeviceGuard g(device);
    H* c = new H(*h);
    c->device = device;
    auto copy = [&](void** dst, const void* src, size_t bytes) -> ndi_status {
        CK(cudaMalloc(dst, bytes));
        CK(cudaMemcpyPeer(*dst, device, src, h->device, bytes));
        return NDI_OK;
    };
    const ndi_status st = fill(c, copy);
    if (st != NDI_OK) { destroy(c); return st; }
    *out = c;
    return NDI_OK;
}

extern "C" {

ndi_status ndi_selftest_fdiv(uint32_t a_mant_begin, uint32_t a_mant_count, int32_t a_exp, int32_t b_exp, uint64_t* mismatches) {
    if (!mismatches || a_exp < -126 || a_exp > 127 || b_exp < -126 || b_exp > 127 ||
        (uint64_t)a_mant_begin + a_mant_count > (1u << 23))
        return fail(NDI_INVALID_ARGUMENT, "bad mantissa or exponent range");
    int dev = 0; CK(cudaGetDevice(&dev));
    ndi_status st; Workspace* ws = workspace(dev, &st); if (!ws) return st;
    CK(cudaMemsetAsync(ws->d_err, 0, sizeof(uint64_t), ws->s[0]));
    CK(launch_selftest_fdiv(a_mant_begin, a_mant_count, a_exp, b_exp, ws->d_err, ws->s[0]));
    CK(cudaMemcpyAsync(ws->h_pin, ws->d_err, sizeof(uint64_t), cudaMemcpyDeviceToHost, ws->s[0]));
    CK(cudaStreamSynchronize(ws->s[0]));
    memcpy(mismatches, ws->h_pin, sizeof(uint64_t));
    return NDI_OK;
}

ndi_status ndi_selftest_ddiv(uint64_t seed, uint64_t pairs, uint64_t* mismatches) {
    if (!mismatches) return fail(NDI_INVALID_ARGUMENT, "null pointer");
    int dev = 0; CK(cudaGetDevice(&dev));
    ndi_status st; Workspace* ws = workspace(dev, &st); if (!ws) return st;
    const int per_thread = 64;                                   // x 8 numerators each
    uint64_t blocks = (pairs + 256ull * per_thread * 8 - 1) / (256ull * per_thread * 8);
    if (blocks < 1) blocks = 1;
    if (blocks > (1u << 30)) return fail(NDI_INVALID_ARGUMENT, "too many pairs");
    CK(cudaMemsetAsync(ws->d_err, 0, sizeof(uint64_t), ws->s[0]));
    CK(launch_selftest_ddiv(seed, (int)blocks, per_thread, ws->d_err, ws->s[0]));
    CK(cudaMemcpyAsync(ws->h_pin, ws->d_err, sizeof(uint64_t), cudaMemcpyDeviceToHost, ws->s[0]));
    CK(cudaStreamSynchronize(ws->s[0]));
    memcpy(mismatches, ws->h_pin, sizeof(uint64_t));
    return NDI_OK;
}

const char* ndi_version_string(void) { return "ndarray-interp-b200 0.1 (sm_100a)"; }
const char* ndi_last_error_message(void) { return g_err; }
uint64_t ndi_kernel_launch_count(void) { return g_launches.load(); }

ndi_status ndi_device_count(int32_t* count) {
    int c = 0;
    cudaError_t e = cudaGetDeviceCount(&c);
    if (e != cudaSuccess) { *count = 0; return cuda_fail(e, "cudaGetDeviceCount"); }
    *count = c;
    return c > 0 ? NDI_OK : fail(NDI_NO_DEVICE, "no CUDA device: this library has no CPU fallback");
}
ndi_status ndi_set_device(int32_t device) { CK(cudaSetDevice(device)); return NDI_OK; }
ndi_status ndi_get_device(int32_t* device) { int d = 0; CK(cudaGetDevice(&d)); *device = d; return NDI_OK; }

// ---- vector_extensions --------------------------------------------------------------------------------------
ndi_status ndi_monotonic_prop(ndi_dtype dtype, const void* x, int64_t n, int64_t stride, int32_t* prop) {
    if (!dtype_ok(dtype)) return fail(NDI_UNSUPPORTED_DTYPE, "unsupported dtype %d", (int)dtype);
    if (!prop || (n > 0 && !x)) return fail(NDI_INVALID_ARGUMENT, "null pointer");
    *prop = NDI_MONO_NOT_MONOTONIC;
    if (n <= 1) return NDI_OK;                                   // vector_extensions.rs:41-43
    int dev = 0; CK(cudaGetDevice(&dev));
    ndi_status st; Workspace* ws = workspace(dev, &st); if (!ws) return st;
    const size_t es = elem_size(dtype), bytes = (size_t)n * es;
    // a strided (possibly reversed) view is made contiguous on the way to the device
    std::vector<unsigned char> packed;
    const void* src = x;
    if (stride != 1) {
        packed.resize(bytes);
        for (int64_t i = 0; i < n; ++i) memcpy(packed.data() + (size_t)i * es, (const unsigned char*)x + i * stride * (int64_t)es, es);
        src = packed.data();
    }
    if ((st = grow(&ws->d_q[0], &ws->d_q_cap[0], bytes)) != NDI_OK) return st;
    CK(cudaMemcpyAsync(ws->d_q[0], src, bytes, cudaMemcpyHostToDevice, ws->s[0]));
    int32_t res[2];
    if ((st = classify_grid(dtype, ws->d_q[0], n, ws, res)) != NDI_OK) return st;
    *prop = res[0];
    return NDI_OK;
}

ndi_status ndi_lower_index_dev(ndi_dtype dtype, const void* grid_dev, int64_t n, const void* q_dev, int64_t nq,
                               int64_t* idx_dev, uint64_t* err_word_dev, int32_t search_mode, void* stream) {
    if (n < 2) return fail(NDI_INVALID_ARGUMENT, "grid needs at least 2 points, got %lld", (long long)n);
    if (n > 0x7fffffffll) return fail(NDI_INVALID_ARGUMENT, "grid longer than 2^31-1");
    cudaStream_t st = (cudaStream_t)stream;
    if (err_word_dev) CK(cudaMemsetAsync(err_word_dev, 0xff, sizeof(uint64_t), st));
    return dispatch(dtype, [&](auto tag) -> ndi_status {
        using T = decltype(tag);
        SearchCfg sc = make_search(GridMeta{grid_dev, n, sizeof(T), 0, nullptr, 0, 0, nullptr, 0, 0.0, 0.0}, search_mode, nq, 0);
        CK(launch_lower_index<T>((const T*)grid_dev, n, sc, (const T*)q_dev, nq, idx_dev, (unsigned long long*)err_word_dev, st));
        return NDI_OK;
    });
}

ndi_status ndi_lower_index(ndi_dtype dtype, const void* grid, int64_t n, const void* q, int64_t nq, int64_t* idx,
                           int64_t* first_bad) {
    if (!dtype_ok(dtype)) return fail(NDI_UNSUPPORTED_DTYPE, "unsupported dtype %d", (int)dtype);
    if (first_bad) *first_bad = -1;
    if (nq <= 0) return NDI_OK;
    if (!grid || !q || !idx) return fail(NDI_INVALID_ARGUMENT, "null pointer");
    int dev = 0; CK(cudaGetDevice(&dev));
    ndi_status st; Workspace* ws = workspace(dev, &st); if (!ws) return st;
    const size_t es = elem_size(dtype);
    if ((st = grow(&ws->d_q[0], &ws->d_q_cap[0], (size_t)nq * es)) != NDI_OK) return st;
    if ((st = grow(&ws->d_q[1], &ws->d_q_cap[1], (size_t)n * es)) != NDI_OK) return st;
    if ((st = grow(&ws->d_out[0], &ws->d_out_cap[0], (size_t)nq * sizeof(int64_t))) != NDI_OK) return st;
    CK(cudaMemcpyAsync(ws->d_q[1], grid, (size_t)n * es, cudaMemcpyHostToDevice, ws->s[0]));
    CK(cudaMemcpyAsync(ws->d_q[0], q, (size_t)nq * es, cudaMemcpyHostToDevice, ws->s[0]));
    st = ndi_lower_index_dev(dtype, ws->d_q[1], n, ws->d_q[0], nq, (int64_t*)ws->d_out[0], (uint64_t*)ws->d_err, NDI_SEARCH_AUTO, ws->s[0]);
    if (st != NDI_OK) return st;
    CK(cudaMemcpyAsync(ws->h_pin, ws->d_err, sizeof(uint64_t), cudaMemcpyDeviceToHost, ws->s[0]));
    CK(cudaStreamSynchronize(ws->s[0]));
    uint64_t word; memcpy(&word, ws->h_pin, sizeof(word));
    const int64_t nvalid = word == NDI_ERR_WORD_NONE ? nq : (int64_t)word;
    if (nvalid > 0) {
        CK(cudaMemcpyAsync(idx, ws->d_out[0], (size_t)nvalid * sizeof(int64_t), cudaMemcpyDeviceToHost, ws->s[0]));
        CK(cudaStreamSynchronize(ws->s[0]));
    }
    if (word != NDI_ERR_WORD_NONE) {
        if (first_bad) *first_bad = (int64_t)word;
        return fail(NDI_NAN_QUERY, "not implemented: failed to convert NaN to usize (query %lld)", (long long)word);
    }
    return NDI_OK;
}

// ---- Interp1D ------------------------------------------------------------------------------------------------
ndi_status ndi_interp1d_create(ndi_dtype dtype, const void* x, int64_t n, const void* data, int64_t w, uint32_t flags,
                               ndi_interp1d** out) {
    if (!out) return fail(NDI_INVALID_ARGUMENT, "null handle pointer");
    *out = nullptr;
    if (!dtype_ok(dtype)) return fail(NDI_UNSUPPORTED_DTYPE, "unsupported dtype %d", (int)dtype);
    if (!x || !data) return fail(NDI_INVALID_ARGUMENT, "null pointer");
    if (n < 2 || w < 1) return fail(NDI_INVALID_ARGUMENT, "need n >= 2 and w >= 1, got n=%lld w=%lld", (long long)n, (long long)w);
    if (n > 0x7fffffffll) return fail(NDI_INVALID_ARGUMENT, "grid longer than 2^31-1");
    int dev = 0; CK(cudaGetDevice(&dev));
    ndi_status st; Workspace* ws = workspace(dev, &st); if (!ws) return st;
    const size_t es = elem_size(dtype);
    ndi_interp1d* h = new ndi_interp1d();
    h->dtype = dtype; h->device = dev; h->n = n; h->w = w;
    h->x = h->data = h->a = h->b = nullptr; h->owns_tables = h->owns_coeffs = false;
    h->uniform_hint = 0; h->search_mode = NDI_SEARCH_AUTO;
    bool ox = false, od = false;
    if ((st = take_table(x, (size_t)n * es, flags, ws->s[0], &h->x, &ox)) != NDI_OK) { delete h; return st; }
    if ((st = take_table(data, (size_t)n * (size_t)w * es, flags, ws->s[0], &h->data, &od)) != NDI_OK) {
        if (ox) cudaFree(h->x);
        delete h; return st;
    }
    h->owns_tables = ox;
    int32_t res[2] = {0, 0};
    st = classify_grid(dtype, h->x, n, ws, res);           // also drains the upload
    if (st == NDI_OK && !(flags & NDI_ASSUME_VALID) && res[0] != NDI_MONO_RISING_STRICT)
        st = fail(NDI_NOT_MONOTONIC, "Values in the x axis need to be strictly monotonic rising");
    if (st != NDI_OK) { ndi_interp1d_destroy(h); return st; }
    h->uniform_hint = res[0] == NDI_MONO_RISING_STRICT ? res[1] : 0;
    if (!h->uniform_hint) {
        st = build_aids(dtype, h->x, n, ws->s[0], &h->aids);
        if (st != NDI_OK) { ndi_interp1d_destroy(h); return st; }
    }
    if ((st = scan_fast_tables(dtype, h->data, (size_t)n * (size_t)w, ws, &h->fast_tables)) != NDI_OK) { ndi_interp1d_destroy(h); return st; }
    if ((st = build_pair_table(h, ws->s[0])) != NDI_OK) { ndi_interp1d_destroy(h); return st; }
    *out = h;
    return NDI_OK;
}

ndi_status ndi_interp1d_create_strided(ndi_dtype dtype, const void* x, int64_t n, int64_t x_stride, const void* data,
                                       int32_t ndim, const int64_t* shape, const int64_t* strides, uint32_t flags,
                                       ndi_interp1d** out) {
    if (!out) return fail(NDI_INVALID_ARGUMENT, "null handle pointer");
    *out = nullptr;
    if (!dtype_ok(dtype)) return fail(NDI_UNSUPPORTED_DTYPE, "unsupported dtype %d", (int)dtype);
    if (!x || !data || !shape || !strides) return fail(NDI_INVALID_ARGUMENT, "null pointer");
    if (flags & NDI_BORROW) return fail(NDI_INVALID_ARGUMENT, "a strided view cannot be borrowed: the kernels read dense tables");
    if (ndim < 1 || ndim > kMaxDims) return fail(NDI_INVALID_ARGUMENT, "data needs 1..%d dimensions", kMaxDims);
    if (shape[0] != n) return fail(NDI_INVALID_ARGUMENT, "data.shape[0] = %lld but x has %lld elements", (long long)shape[0], (long long)n);
    int dev = 0; CK(cudaGetDevice(&dev));
    ndi_status st; Workspace* ws = workspace(dev, &st); if (!ws) return st;
    const size_t es = elem_size(dtype);
    const bool dsrc = (flags & NDI_DEVICE_POINTERS) != 0;
    int64_t w = 1;
    for (int k = 1; k < ndim; ++k) w *= shape[k];
    void *xd = nullptr, *dd = nullptr;
    if ((st = pack_view(x, es, 1, &n, &x_stride, dsrc, ws->s[0], &xd)) != NDI_OK) return st;
    if ((st = pack_view(data, es, ndim, shape, strides, dsrc, ws->s[0], &dd)) != NDI_OK) { cudaFree(xd); return st; }
    st = ndi_interp1d_create(dtype, xd, n, dd, w, (flags & NDI_ASSUME_VALID) | NDI_DEVICE_POINTERS | NDI_BORROW, out);
    if (st != NDI_OK) { cudaFree(xd); cudaFree(dd); return st; }
    (*out)->owns_tables = true;                            // the dense copies belong to the handle
    return NDI_OK;
}

ndi_status ndi_interp1d_destroy(ndi_interp1d* h) {
    if (!h) return NDI_OK;
    DeviceGuard g(h->device);
    if (h->owns_tables) { cudaFree(h->x); cudaFree(h->data); }
    if (h->owns_coeffs) { cudaFree(h->a); cudaFree(h->b); }
    cudaFree(h->pair);
    h->aids.release();
    delete h;
    return NDI_OK;
}

ndi_status ndi_interp1d_info(const ndi_interp1d* h, ndi_dtype* dtype, int64_t* n, int64_t* w, int32_t* has_spline, int32_t* device) {
    if (!h) return fail(NDI_INVALID_ARGUMENT, "null handle");
    if (dtype) *dtype = h->dtype;
    if (n) *n = h->n;
    if (w) *w = h->w;
    if (has_spline) *has_spline = h->a != nullptr;
    if (device) *device = h->device;
    return NDI_OK;
}
ndi_status ndi_interp1d_set_search_mode(ndi_interp1d* h, int32_t mode) {
    if (!h || mode < 0 || mode > NDI_SEARCH_MERGE) return fail(NDI_INVALID_ARGUMENT, "bad search mode");
    h->search_mode = mode;
    return NDI_OK;
}
ndi_status ndi_interp1d_device_ptrs(const ndi_interp1d* h, const void** x, const void** data, const void** a, const void** b) {
    if (!h) return fail(NDI_INVALID_ARGUMENT, "null handle");
    if (x) *x = h->x;
    if (data) *data = h->data;
    if (a) *a = h->a;
    if (b) *b = h->b;
    return NDI_OK;
}

ndi_status ndi_interp1d_clone_to_device(const ndi_interp1d* h, int32_t device, ndi_interp1d** out) {
    return clone_to_device(h, device, out, ndi_interp1d_destroy, [&](ndi_interp1d* c, auto& copy) {
        const size_t es = elem_size(h->dtype);
        c->owns_tables = true; c->owns_coeffs = h->a != nullptr;
        c->x = c->data = c->a = c->b = c->pair = nullptr;
        c->aids = GridAids{};
        ndi_status st = copy(&c->x, h->x, (size_t)h->n * es);
        if (st == NDI_OK) st = copy(&c->data, h->data, (size_t)h->n * h->w * es);
        if (st == NDI_OK && h->a) st = copy(&c->a, h->a, (size_t)(h->n - 1) * h->w * es);
        if (st == NDI_OK && h->b) st = copy(&c->b, h->b, (size_t)(h->n - 1) * h->w * es);
        if (st == NDI_OK && !h->uniform_hint) st = build_aids(c->dtype, c->x, c->n, nullptr, &c->aids);
        if (st == NDI_OK && h->pair) st = copy(&c->pair, h->pair, (size_t)(h->n - 1) * 2 * h->w * es);
        return st;
    });
}

}  // extern "C"

// ---- host-buffer pipeline -----------------------------------------------------------------------------------
namespace {

// A batch fanned out over several devices (ndi_*_group_*) runs each device's block of queries in two calls on the
// block's worker thread, because the reference stops at the first failing query of the WHOLE batch.
enum class Phase {
    whole,      // everything in one call
    prepass,    // queries up, pre-pass: *err_word = first failing query of this block
    evaluate,   // evaluate the first `nvalid` rows only (the caller knows the batch-wide first failure by now)
};

struct HostEval {
    int device; size_t es; int ncoord; int64_t w;
    const void* q[2]; int64_t nq; void* out;
    // launch(q0_dev, q1_dev, nq, out_dev, err_dev, stream) evaluates a contiguous range of queries
    // validate(q0_dev, q1_dev, nq, err_dev, stream) is the K7 pre-pass over a contiguous range of queries
    Phase phase;
    int64_t nvalid;           // Phase::evaluate
};

// An error word is the index of the first failing query (2-D: 2 * index + axis) within the range it was taken over.
inline int64_t err_query(uint64_t word, int ncoord) { return (int64_t)(ncoord > 1 ? word >> 1 : word); }
// ... and, for a range that starts at query `lo`, this is the same word within the whole batch
inline uint64_t err_rebase(uint64_t word, int ncoord, int64_t lo) { return word + (ncoord > 1 ? 2 : 1) * (uint64_t)lo; }

template <class Launch, class Validate>
ndi_status run_host_eval(const HostEval& he, Launch&& launch, Validate&& validate, uint64_t* err_word) {
    *err_word = NDI_ERR_WORD_NONE;
    if (he.nq <= 0) return NDI_OK;
    DeviceGuard g(he.device);
    ndi_status st; Workspace* ws = workspace(he.device, &st); if (!ws) return st;
    const size_t qbytes = (size_t)he.nq * he.es;
    const size_t row = (size_t)he.w * he.es;
    const size_t total = (size_t)he.nq * row;
    if (he.phase == Phase::whole && total <= kTinyBytes) {
        // scalar / tiny-batch latency path (interp_scalar, interp, interp_into: interp1d/mod.rs:108-175): the
        // pinned workspace is mapped into the device's address space, so the kernel reads the queries from
        // it and writes the rows into it over PCIe; publish_kernel hands over the error word and raises the
        // flag this thread spins on: two launches, no copy call, no driver synchronisation
        unsigned char* hq0 = ws->h_pin + 64 + kTinyBytes;
        unsigned char* hq1 = hq0 + kTinyBytes;
        memcpy(hq0, he.q[0], qbytes);
        if (he.ncoord > 1) memcpy(hq1, he.q[1], qbytes);
        unsigned long long* tiny_err = ws->d_err + 1;          // its own word: publish_kernel leaves it armed (~0)
        if (!ws->err_armed) { CK(cudaMemsetAsync(tiny_err, 0xff, sizeof(uint64_t), ws->s[0])); ws->err_armed = true; }
        if ((st = launch(hq0, he.ncoord > 1 ? hq1 : nullptr, he.nq, ws->h_pin + 64, tiny_err, ws->s[0])) != NDI_OK) return st;
        const unsigned long long seq = ++ws->seq;
        volatile unsigned long long* flag = reinterpret_cast<volatile unsigned long long*>(ws->h_pin + 8);
        CK(launch_publish(tiny_err, ws->h_pin, ws->h_pin + 8, seq, ws->s[0]));
        for (unsigned spins = 1; *flag != seq; ++spins) {       // the kernels raise the flag; the driver is asked only now and then
            if ((spins & 0x3fff) == 0) {
                const cudaError_t q = cudaStreamQuery(ws->s[0]);
                if (q != cudaSuccess && q != cudaErrorNotReady) return cuda_fail(q, "tiny-batch evaluation");
            }
#if defined(__x86_64__)
            __builtin_ia32_pause();
#endif
        }
        std::atomic_thread_fence(std::memory_order_acquire);
        memcpy(err_word, ws->h_pin, sizeof(uint64_t));
        const int64_t nvalid = *err_word == NDI_ERR_WORD_NONE ? he.nq : err_query(*err_word, he.ncoord);
        memcpy(he.out, ws->h_pin + 64, (size_t)nvalid * row);
        return NDI_OK;
    }
    unsigned long long* d_err = ws->d_err;
    for (int c = 0; c < he.ncoord && he.phase != Phase::evaluate; ++c)   // Phase::evaluate: this thread's prepass uploaded them
        if ((st = grow(&ws->d_q[c], &ws->d_q_cap[c], qbytes)) != NDI_OK) return st;
    const void* dq0 = ws->d_q[0];
    const void* dq1 = he.ncoord > 1 ? ws->d_q[1] : nullptr;

    if (he.phase == Phase::prepass) {                            // K7 pre-pass over the whole block: where would the reference stop?
        auto prepass = [&]() -> ndi_status {
            for (int c = 0; c < he.ncoord; ++c) CK(cudaMemcpyAsync(ws->d_q[c], he.q[c], qbytes, cudaMemcpyHostToDevice, ws->s[0]));
            CK(cudaMemsetAsync(d_err, 0xff, sizeof(uint64_t), ws->s[0]));
            if ((st = validate(dq0, dq1, he.nq, d_err, ws->s[0])) != NDI_OK) return st;
            CK(cudaMemcpyAsync(ws->h_pin, d_err, sizeof(uint64_t), cudaMemcpyDeviceToHost, ws->s[0]));
            CK(cudaStreamSynchronize(ws->s[0]));
            memcpy(err_word, ws->h_pin, sizeof(uint64_t));
            return NDI_OK;
        };
        if ((st = prepass()) != NDI_OK) cudaStreamSynchronize(ws->s[0]);   // no upload from the caller's memory left in flight
        return st;
    }

    // A whole call over a large batch STREAMS: the queries go up chunk by chunk on a copy-in stream, a few chunks ahead
    // of the evaluation, each followed by the pre-pass over that chunk, so the upload (host -> device) runs beside the
    // copy-out of earlier chunks (device -> host) instead of in front of it -- PCIe is full duplex, and for thin rows
    // the queries are a fifth of the bytes on the link (C4: 134 MB up, 537 MB down).  Chunks are consumed in order, so
    // stopping at the first chunk whose pre-pass reports a failure is the reference's "first Err" exactly.
    const bool streaming = he.phase == Phase::whole;
    const int64_t nvalid = streaming ? he.nq : (he.nvalid < he.nq ? he.nvalid : he.nq);
    if (nvalid <= 0) return NDI_OK;

    // Where finished chunks go: page-locked memory (or rows too wide to stage) receives them straight from the device;
    // ordinary pageable memory through three pinned staging buffers, which the copy pool empties into it.
    const bool staged = row <= kStageBytes / 32 && is_pageable_host(he.out);
    int64_t per = (int64_t)((staged ? kStageBytes : kChunkBytes) / row) & ~31ll;   // queries per chunk
    if (per < 32) per = 32;
    const size_t chunk_bytes = (size_t)per * row;
    CopyPool* pool = nullptr;
    uint64_t ticket[3] = {0, 0, 0};
    int64_t staged_cnt[3] = {0, 0, 0};
    if (staged) {
        for (int k = 0; k < 3; ++k) {
            if (!ws->h_stage[k]) CK(cudaMallocHost(&ws->h_stage[k], kStageBytes));
            if (!ws->stage_ev[k]) CK(cudaEventCreateWithFlags(&ws->stage_ev[k], cudaEventDisableTiming));
        }
        pool = &CopyPool::get();
    }
    auto hand_over = [&](int64_t j) -> ndi_status {             // chunk j has landed in its staging buffer: hand it to the pool
        const int k = (int)(j % 3);
        CK(cudaEventSynchronize(ws->stage_ev[k]));
        ticket[k] = pool->submit((unsigned char*)he.out + (size_t)(j * per) * row, ws->h_stage[k], (size_t)staged_cnt[k] * row);
        return NDI_OK;
    };

    // the copy-in side of the streaming pipeline: chunk i = queries [i * per, (i + 1) * per)
    constexpr int kFeedDepth = 3;
    auto feed = [&](int64_t i) -> ndi_status {
        const int64_t lo = i * per;
        if (!streaming || lo >= he.nq) return NDI_OK;
        const int64_t cnt = he.nq - lo < per ? he.nq - lo : per;
        const int k = (int)(i % kFeedDepth);
        for (int c = 0; c < he.ncoord; ++c)
            CK(cudaMemcpyAsync((unsigned char*)ws->d_q[c] + (size_t)lo * he.es, (const unsigned char*)he.q[c] + (size_t)lo * he.es,
                               (size_t)cnt * he.es, cudaMemcpyHostToDevice, ws->s_in));
        CK(cudaMemsetAsync(d_err + 4 + k, 0xff, sizeof(uint64_t), ws->s_in));
        ndi_status fs = validate((const unsigned char*)dq0 + (size_t)lo * he.es, dq1 ? (const unsigned char*)dq1 + (size_t)lo * he.es : nullptr,
                                 cnt, d_err + 4 + k, ws->s_in);
        if (fs != NDI_OK) return fs;
        CK(cudaMemcpyAsync(ws->h_pin + 16 + 8 * k, d_err + 4 + k, sizeof(uint64_t), cudaMemcpyDeviceToHost, ws->s_in));
        CK(cudaEventRecord(ws->feed_ev[k], ws->s_in));
        return NDI_OK;
    };
    // chunk i has arrived: how many of its rows does the reference write?  (fewer than all: the batch ends there)
    auto fed = [&](int64_t i, int64_t cnt, int64_t* cnt_valid) -> ndi_status {
        *cnt_valid = cnt;
        if (!streaming) return NDI_OK;
        const int k = (int)(i % kFeedDepth);
        CK(cudaEventSynchronize(ws->feed_ev[k]));
        uint64_t word; memcpy(&word, ws->h_pin + 16 + 8 * k, sizeof(word));
        if (word != NDI_ERR_WORD_NONE) {
            *cnt_valid = err_query(word, he.ncoord);
            *err_word = err_rebase(word, he.ncoord, i * per);
        }
        return NDI_OK;
    };

    st = NDI_OK;
    for (int64_t i = 0; i < kFeedDepth && st == NDI_OK; ++i) st = feed(i);
    int64_t launched = 0;                                        // chunks whose copy-out was issued
    for (int64_t i = 0; i * per < nvalid && st == NDI_OK; ++i) {
        const int64_t lo = i * per, full = nvalid - lo < per ? nvalid - lo : per;
        const int slot = (int)(i & 1), k = (int)(i % 3);
        int64_t cnt;
        if ((st = fed(i, full, &cnt)) != NDI_OK) break;
        if ((st = feed(i + kFeedDepth)) != NDI_OK) break;
        if (staged) pool->wait(ticket[k]);                       // the host copy that last used this staging buffer is done
        if (cnt > 0) {
            if ((st = grow(&ws->d_out[slot], &ws->d_out_cap[slot], chunk_bytes < total ? chunk_bytes : total)) != NDI_OK) break;
            const void* c0 = (const unsigned char*)dq0 + (size_t)lo * he.es;
            const void* c1 = dq1 ? (const unsigned char*)dq1 + (size_t)lo * he.es : nullptr;
            if ((st = launch(c0, c1, cnt, ws->d_out[slot], nullptr, ws->s[slot])) != NDI_OK) break;
            void* dst = staged ? (void*)ws->h_stage[k] : (void*)((unsigned char*)he.out + (size_t)lo * row);
            cudaError_t ce = cudaMemcpyAsync(dst, ws->d_out[slot], (size_t)cnt * row, cudaMemcpyDeviceToHost, ws->s[slot]);
            if (ce == cudaSuccess && staged) ce = cudaEventRecord(ws->stage_ev[k], ws->s[slot]);
            if (ce != cudaSuccess) { st = cuda_fail(ce, staged ? "staged copy" : "copy-out"); break; }
            staged_cnt[k] = cnt;
            if (staged && launched >= 1) st = hand_over(launched - 1);
            ++launched;
        }
        if (cnt < full) break;                                   // the reference stopped inside this chunk
    }
    if (staged) {
        if (st == NDI_OK && launched >= 1) st = hand_over(launched - 1);
        for (uint64_t t : ticket) pool->wait(t);
    }
    // never return while a copy from (or into) the caller's memory is in flight
    if (st != NDI_OK) {
        if (streaming) cudaStreamSynchronize(ws->s_in);
        cudaStreamSynchronize(ws->s[0]); cudaStreamSynchronize(ws->s[1]);
        return st;
    }
    if (streaming) CK(cudaStreamSynchronize(ws->s_in));
    CK(cudaStreamSynchronize(ws->s[0]));
    CK(cudaStreamSynchronize(ws->s[1]));
    return NDI_OK;
}

// one evaluation of a device-resident batch, for the _dev entry points and the host pipeline
template <class T>
ndi_status linear_on_device(const ndi_interp1d* h, const SearchCfg& sc, const T* q, int64_t nq, int extrapolate, T* out,
                            unsigned long long* err, cudaStream_t s) {
    CK(launch_interp1d_linear<T>((const T*)h->x, h->n, sc, (const T*)h->data, h->w, q, nq, extrapolate != 0, out, err,
                                 h->fast_tables, (const T*)h->pair, s));
    return NDI_OK;
}
template <class T>
ndi_status cubic_on_device(const ndi_interp1d* h, const SearchCfg& sc, const T* q, int64_t nq, int extrap_mode, T* out,
                           unsigned long long* err, cudaStream_t s) {
    CK(launch_interp1d_cubic<T>((const T*)h->x, h->n, sc, (const T*)h->data, (const T*)h->a, (const T*)h->b, h->w, q, nq,
                                extrap_mode, out, err, s));
    return NDI_OK;
}
// derivatives (NOT in the reference): the same query handling, K3d / K5d per element
template <class T>
ndi_status linear_deriv_on_device(const ndi_interp1d* h, const SearchCfg& sc, const T* q, int64_t nq, int extrapolate, T* out,
                                  unsigned long long* err, cudaStream_t s) {
    CK(launch_interp1d_linear_slope<T>((const T*)h->x, h->n, sc, (const T*)h->data, h->w, q, nq, extrapolate != 0, out, err, s));
    return NDI_OK;
}
template <class T>
ndi_status cubic_deriv_on_device(const ndi_interp1d* h, const SearchCfg& sc, const T* q, int64_t nq, int extrap_mode, int order,
                                 T* out, unsigned long long* err, cudaStream_t s) {
    CK(launch_interp1d_cubic_deriv<T>((const T*)h->x, h->n, sc, (const T*)h->data, (const T*)h->a, (const T*)h->b, h->w, q, nq,
                                      extrap_mode, order, out, err, s));
    return NDI_OK;
}

}  // namespace

extern "C" {

static ndi_status check_eval_args(const void* h, const void* q, int64_t nq, const void* out) {
    if (!h) return fail(NDI_INVALID_ARGUMENT, "null handle");
    if (nq < 0) return fail(NDI_INVALID_ARGUMENT, "negative query count");
    if (nq > 0 && (!q || !out)) return fail(NDI_INVALID_ARGUMENT, "null pointer");
    return NDI_OK;
}

ndi_status ndi_interp1d_linear_dev(const ndi_interp1d* h, const void* q_dev, int64_t nq, int32_t extrapolate,
                                   void* out_dev, uint64_t* err_word_dev, void* stream) {
    ndi_status st = check_eval_args(h, q_dev, nq, out_dev); if (st != NDI_OK) return st;
    cudaStream_t s = (cudaStream_t)stream;
    if (err_word_dev) CK(cudaMemsetAsync(err_word_dev, 0xff, sizeof(uint64_t), s));
    return dispatch(h->dtype, [&](auto tag) -> ndi_status {
        using T = decltype(tag);
        SearchCfg sc = make_search(h->meta(), h->search_mode, nq, 0);
        return linear_on_device<T>(h, sc, (const T*)q_dev, nq, extrapolate, (T*)out_dev, (unsigned long long*)err_word_dev, s);
    });
}

ndi_status ndi_interp1d_linear_deriv_dev(const ndi_interp1d* h, const void* q_dev, int64_t nq, int32_t extrapolate,
                                         void* out_dev, uint64_t* err_word_dev, void* stream) {
    ndi_status st = check_eval_args(h, q_dev, nq, out_dev); if (st != NDI_OK) return st;
    cudaStream_t s = (cudaStream_t)stream;
    if (err_word_dev) CK(cudaMemsetAsync(err_word_dev, 0xff, sizeof(uint64_t), s));
    return dispatch(h->dtype, [&](auto tag) -> ndi_status {
        using T = decltype(tag);
        SearchCfg sc = make_search(h->meta(), h->search_mode, nq, 0);
        return linear_deriv_on_device<T>(h, sc, (const T*)q_dev, nq, extrapolate, (T*)out_dev, (unsigned long long*)err_word_dev, s);
    });
}

// one block of a host batch (Phase::whole: the whole call); slope: the derivative instead of the values
static ndi_status linear_host(const ndi_interp1d* h, const void* q, int64_t nq, int32_t extrapolate, void* out,
                              uint64_t* word, Phase phase, int64_t nvalid, bool slope = false) {
    HostEval he{h->device, elem_size(h->dtype), 1, h->w, {q, nullptr}, nq, out, phase, nvalid};
    return dispatch(h->dtype, [&](auto tag) -> ndi_status {
        using T = decltype(tag);
        SearchCfg sc = make_search(h->meta(), h->search_mode, nq, 0);
        return run_host_eval(he,
            [&](const void* q0, const void*, int64_t cnt, void* o, unsigned long long* err, cudaStream_t s) -> ndi_status {
                if (slope) return linear_deriv_on_device<T>(h, sc, (const T*)q0, cnt, extrapolate, (T*)o, err, s);
                return linear_on_device<T>(h, sc, (const T*)q0, cnt, extrapolate, (T*)o, err, s);
            },
            [&](const void* q0, const void*, int64_t cnt, unsigned long long* err, cudaStream_t s) -> ndi_status {
                CK(launch_validate_queries<T>((const T*)h->x, h->n, nullptr, 0, (const T*)q0, nullptr, cnt,
                                              extrapolate ? CHECK_NOT_NAN : CHECK_IN_RANGE, err, s));
                return NDI_OK;
            }, word);
    });
}
static ndi_status eval1d_status(uint64_t word, int nan_only, int64_t* first_bad) {
    if (word == NDI_ERR_WORD_NONE) return NDI_OK;
    if (first_bad) *first_bad = (int64_t)word;
    return nan_only ? fail(NDI_NAN_QUERY, "not implemented: failed to convert NaN to usize (query %lld)", (long long)word)
                    : fail(NDI_OUT_OF_BOUNDS, "query %lld is not in range", (long long)word);
}

ndi_status ndi_interp1d_linear(const ndi_interp1d* h, const void* q, int64_t nq, int32_t extrapolate, void* out,
                               int64_t* first_bad) {
    if (first_bad) *first_bad = -1;
    ndi_status st = check_eval_args(h, q, nq, out); if (st != NDI_OK) return st;
    uint64_t word;
    if ((st = linear_host(h, q, nq, extrapolate, out, &word, Phase::whole, 0)) != NDI_OK) return st;
    return eval1d_status(word, extrapolate, first_bad);
}

ndi_status ndi_interp1d_linear_deriv(const ndi_interp1d* h, const void* q, int64_t nq, int32_t extrapolate, void* out,
                                     int64_t* first_bad) {
    if (first_bad) *first_bad = -1;
    ndi_status st = check_eval_args(h, q, nq, out); if (st != NDI_OK) return st;
    uint64_t word;
    if ((st = linear_host(h, q, nq, extrapolate, out, &word, Phase::whole, 0, true)) != NDI_OK) return st;
    return eval1d_status(word, extrapolate, first_bad);
}

// ---- cubic spline ---------------------------------------------------------------------------------------------
// The reference's NotAKnot system takes x[n-1] - x[n-2] for the last diagonal entry (cubic_spline.rs:635, the quirk kept
// on purpose, DESIGN.md section 2).  With that entry the last pivot of the elimination,
//     mid'[n-1] = (x[n-1] - x[n-2]) - (x[n-1] - x[n-3]) / mid'[n-2] * (x[n-2] - x[n-3]),
// vanishes when the last grid step is about 0.55 of the one before it: the reference's own result is then the quotient of
// two rounding errors, and any other order of operations moves it by as much (partition against reference order, f32:
// up to 6e-5 of the column's scale inside |pivot| < 0.03 of the entry, 3e-6 up to 0.1, 1e-6 beyond; profiles/r02/
// partition_build.md).  NDI_BUILD_AUTO therefore keeps the reference's order -- and with it the reference's bits --
// whenever a right NotAKnot row meets such a grid.  The pivot ratio is formed once per handle from the last grid points
// (the elimination forgets its start at a rate of ~0.07 per row; 64 rows are exact to double precision).
constexpr double kNakPivotFloor = 0.1;
static ndi_status nak_pivot_ratio(ndi_interp1d* h, cudaStream_t st, double* ratio) {
    if (h->nak_pivot >= 0.0) { *ratio = h->nak_pivot; return NDI_OK; }
    const int64_t n = h->n, cnt = n < 67 ? n : 67;
    const size_t es = elem_size(h->dtype);
    unsigned char raw[67 * 8];
    CK(cudaMemcpyAsync(raw, (const unsigned char*)h->x + (size_t)(n - cnt) * es, (size_t)cnt * es, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    double x[67];
    for (int64_t i = 0; i < cnt; ++i) {
        if (h->dtype == NDI_F32) { float v; memcpy(&v, raw + i * 4, 4); x[i] = v; }
        else { double v; memcpy(&v, raw + i * 8, 8); x[i] = v; }
    }
    // rows 1 .. cnt-2 of the window are interior rows (:440-451); the first one starts from its own diagonal entry
    double mp = 2.0 * (x[2] - x[0]);
    for (int64_t i = 2; i + 1 < cnt; ++i) mp = 2.0 * (x[i + 1] - x[i - 1]) - (x[i + 1] - x[i]) / mp * (x[i - 1] - x[i - 2]);
    const double mid = x[cnt - 1] - x[cnt - 2], low = x[cnt - 1] - x[cnt - 3], up = x[cnt - 2] - x[cnt - 3];
    double r = fabs(mid - low / mp * up) / fabs(mid);
    if (!(r == r)) r = 0.0;
    h->nak_pivot = r; *ratio = r;
    return NDI_OK;
}

ndi_status ndi_interp1d_spline_build(ndi_interp1d* h, int32_t bc_kind, const int32_t* left_kind, const void* left_val,
                                     const int32_t* right_kind, const void* right_val, int64_t* bad_column) {
    if (bad_column) *bad_column = -1;
    if (!h) return fail(NDI_INVALID_ARGUMENT, "null handle");
    if (bc_kind < NDI_BC_NOT_A_KNOT || bc_kind > NDI_BC_INDIVIDUAL) return fail(NDI_INVALID_ARGUMENT, "bad boundary kind %d", bc_kind);
    if (h->n < 3) return fail(NDI_INVALID_ARGUMENT, "The chosen Interpolation strategy needs at least 3 data points");
    if (bc_kind == NDI_BC_INDIVIDUAL) {
        if (!left_kind || !left_val || !right_kind || !right_val) return fail(NDI_INVALID_ARGUMENT, "Individual boundaries need all four arrays");
        for (int64_t c = 0; c < h->w; ++c)
            if (left_kind[c] < 0 || left_kind[c] > NDI_SB_SECOND_DERIV || right_kind[c] < 0 || right_kind[c] > NDI_SB_SECOND_DERIV)
                return fail(NDI_INVALID_ARGUMENT, "bad single-boundary kind in column %lld", (long long)c);
    }
    DeviceGuard g(h->device);
    ndi_status st; Workspace* ws = workspace(h->device, &st); if (!ws) return st;
    // which solve: the reference's elimination order, or the row-split (PCR + Thomas) build
    const int mode = h->build_mode, want_levels = h->build_levels;
    int levels = 0;
    // AUTO: the partition build from kPartitionAutoRows rows on -- it beats the reference order (serial chains of n steps)
    // and the row-split build at every measured shape from there on, few long columns (4096 x 1024 f64: 0.11 against 0.91
    // and 0.20 ms) as well as many (4096 x 16384 f32: 0.54 against 1.01 and 1.40 ms); at 512 rows the three are level
    // (profiles/r02/partition_build.md).  Shorter systems keep the reference's order and with it the reference's bits.
    bool auto_partition = mode == NDI_BUILD_AUTO && h->n >= kPartitionAutoRows;
    if (auto_partition) {                                     // a NotAKnot row on the right over a grid that makes the reference's system singular?
        bool right_nak = bc_kind == NDI_BC_NOT_A_KNOT;
        if (bc_kind == NDI_BC_INDIVIDUAL)
            for (int64_t c = 0; c < h->w && !right_nak; ++c) right_nak = right_kind[c] == NDI_SB_NOT_A_KNOT;
        if (right_nak && (h->dtype == NDI_F32 || h->dtype == NDI_F64)) {
            double ratio = 1.0;
            ndi_status ps = nak_pivot_ratio(h, ws->s[0], &ratio);
            if (ps != NDI_OK) return ps;
            if (ratio < kNakPivotFloor) auto_partition = false;
        }
    }
    if (h->n >= 4 && (mode == NDI_BUILD_PARTITION || auto_partition))
        levels = -partition_block_for(mode == NDI_BUILD_PARTITION ? want_levels : 0);   // negative: partition build, blocks of that many rows
    else if (h->n >= 4 && mode == NDI_BUILD_ROWSPLIT)
        levels = rowsplit_levels_for(bc_kind == NDI_BC_PERIODIC ? h->n - 2 : h->n, want_levels, true);
    return dispatch_float(h->dtype, [&](auto tag) -> ndi_status {
        using T = decltype(tag);
        const size_t coef_bytes = (size_t)(h->n - 1) * h->w * sizeof(T);
        T *a = nullptr, *b = nullptr, *scratch = nullptr, *lv = nullptr, *rv = nullptr;
        int32_t *lk = nullptr, *rk = nullptr, *pos = nullptr;
        // Individual: group the columns by the kinds of their two boundary rows (what decides the matrix)
        std::vector<int32_t> pos_host;
        int64_t group_count[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
        if (bc_kind == NDI_BC_INDIVIDUAL) {
            auto variant = [](int32_t k) { return k == NDI_SB_NOT_A_KNOT ? 0 : ((k == NDI_SB_FIRST_DERIV || k == NDI_SB_CLAMPED) ? 1 : 2); };
            pos_host.resize((size_t)h->w);
            for (int64_t c = 0; c < h->w; ++c) ++group_count[3 * variant(left_kind[c]) + variant(right_kind[c])];
            int64_t next[9], acc = 0;
            for (int g = 0; g < 9; ++g) { next[g] = acc; acc += group_count[g]; }
            for (int64_t c = 0; c < h->w; ++c) pos_host[(size_t)c] = (int32_t)next[3 * variant(left_kind[c]) + variant(right_kind[c])]++;
        }
        // The scratch matrix and the per-column boundary arrays live in one per-thread buffer that is kept between
        // builds: taken from the stream-ordered pool instead, the wall time of a build depended on the pool's
        // history (scripts/probe_spline_calls.py: the first four calls on a new handle 2 - 10 x slower, 61 ms
        // outliers when consecutive builds asked for different sizes).  a / b come from the pool: they outlive
        // the call, and the previous pair must stay valid until this build has succeeded.
        cudaStream_t bs = ws->s[0];
        constexpr size_t kBuildKeepBytes = (size_t)1 << 30;
        void* big_scratch = nullptr;
        auto cleanup = [&](bool keep) {
            if (big_scratch) { cudaFreeAsync(big_scratch, bs); big_scratch = nullptr; }
            if (!keep) { cudaFreeAsync(a, bs); cudaFreeAsync(b, bs); }
            cudaGetLastError();
        };
        auto body = [&]() -> ndi_status {
            device_info();
            auto up = [](size_t v) { return (v + 255) & ~(size_t)255; };
            const size_t scratch_bytes = up(spline_scratch_elems<T>(h->n, h->w, bc_kind, levels) * sizeof(T));
            const size_t col_i = up((size_t)h->w * sizeof(int32_t)), col_t = up((size_t)h->w * sizeof(T));
            const size_t need = scratch_bytes + (bc_kind == NDI_BC_INDIVIDUAL ? 3 * col_i + 2 * col_t : 0);
            unsigned char* base;
            if (need > kBuildKeepBytes) {
                // beyond what a thread keeps for itself: from the stream-ordered pool, which caches the block between
                // builds (cudaMalloc + cudaFree of 2 GB per call cost 20 ms of a 33 ms build, profiles/r02)
                CK(cudaMallocAsync(&big_scratch, need, bs));
                base = static_cast<unsigned char*>(big_scratch);
            } else {
                ndi_status gs = grow(&ws->d_build, &ws->d_build_cap, need);
                if (gs != NDI_OK) return gs;
                base = static_cast<unsigned char*>(ws->d_build);
            }
            scratch = reinterpret_cast<T*>(base);
            CK(cudaMallocAsync((void**)&a, coef_bytes, bs));
            CK(cudaMallocAsync((void**)&b, coef_bytes, bs));
            if (bc_kind == NDI_BC_INDIVIDUAL) {
                lk = reinterpret_cast<int32_t*>(base + scratch_bytes); rk = reinterpret_cast<int32_t*>(base + scratch_bytes + col_i);
                pos = reinterpret_cast<int32_t*>(base + scratch_bytes + 2 * col_i);
                lv = reinterpret_cast<T*>(base + scratch_bytes + 3 * col_i); rv = reinterpret_cast<T*>(base + scratch_bytes + 3 * col_i + col_t);
                CK(cudaMemcpyAsync(lk, left_kind, h->w * sizeof(int32_t), cudaMemcpyHostToDevice, bs));
                CK(cudaMemcpyAsync(rk, right_kind, h->w * sizeof(int32_t), cudaMemcpyHostToDevice, bs));
                CK(cudaMemcpyAsync(lv, left_val, h->w * sizeof(T), cudaMemcpyHostToDevice, bs));
                CK(cudaMemcpyAsync(rv, right_val, h->w * sizeof(T), cudaMemcpyHostToDevice, bs));
                CK(cudaMemcpyAsync(pos, pos_host.data(), h->w * sizeof(int32_t), cudaMemcpyHostToDevice, bs));
            }
            // the error word (first column whose ends differ) only exists for Periodic: the other kinds save its round trip
            const bool has_err = bc_kind == NDI_BC_PERIODIC;
            if (has_err) CK(cudaMemsetAsync(ws->d_err, 0xff, sizeof(uint64_t), bs));
            CK(launch_spline_build<T>((const T*)h->x, h->n, (const T*)h->data, h->w, bc_kind, lk, lv, rk, rv, pos, group_count, levels, a, b, scratch, ws->d_err, bs));
            if (has_err) CK(cudaMemcpyAsync(ws->h_pin, ws->d_err, sizeof(uint64_t), cudaMemcpyDeviceToHost, bs));
            else { const uint64_t none = NDI_ERR_WORD_NONE; memcpy(ws->h_pin, &none, sizeof(none)); }
            CK(cudaStreamSynchronize(bs));
            return NDI_OK;
        };
        ndi_status s2 = body();
        if (s2 != NDI_OK) { cleanup(false); return s2; }
        uint64_t word; memcpy(&word, ws->h_pin, sizeof(word));
        if (word != NDI_ERR_WORD_NONE) {
            cleanup(false);
            if (bad_column) *bad_column = (int64_t)word;
            return fail(NDI_PERIODIC_MISMATCH, "for periodic boundary condition the first and last value must be equal (column %lld)", (long long)word);
        }
        cleanup(true);
        if (h->owns_coeffs) { cudaFreeAsync(h->a, bs); cudaFreeAsync(h->b, bs); }
        h->a = a; h->b = b; h->owns_coeffs = true;
        h->built_levels = levels;
        return NDI_OK;
    });
}

ndi_status ndi_interp1d_set_build_mode(ndi_interp1d* h, int32_t mode, int32_t levels) {
    if (!h || mode < NDI_BUILD_AUTO || mode > NDI_BUILD_PARTITION || levels < 0) return fail(NDI_INVALID_ARGUMENT, "bad build mode");
    h->build_mode = mode; h->build_levels = levels;
    return NDI_OK;
}
ndi_status ndi_interp1d_build_info(const ndi_interp1d* h, int32_t* rowsplit_levels) {
    if (!h || !rowsplit_levels) return fail(NDI_INVALID_ARGUMENT, "null pointer");
    if (h->built_levels == kNotBuilt) return fail(NDI_NO_SPLINE, "no spline coefficients built by this handle");
    *rowsplit_levels = h->built_levels;
    return NDI_OK;
}

ndi_status ndi_interp1d_spline_coeffs(const ndi_interp1d* h, void* a, void* b) {
    if (!h || !a || !b) return fail(NDI_INVALID_ARGUMENT, "null pointer");
    if (!h->a) return fail(NDI_NO_SPLINE, "no spline coefficients: call ndi_interp1d_spline_build first");
    DeviceGuard g(h->device);
    const size_t bytes = (size_t)(h->n - 1) * h->w * elem_size(h->dtype);
    CK(cudaMemcpy(a, h->a, bytes, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(b, h->b, bytes, cudaMemcpyDeviceToHost));
    return NDI_OK;
}

ndi_status ndi_interp1d_spline_set_coeffs(ndi_interp1d* h, const void* a, const void* b, uint32_t flags) {
    if (!h || !a || !b) return fail(NDI_INVALID_ARGUMENT, "null pointer");
    if (h->dtype != NDI_F32 && h->dtype != NDI_F64) return fail(NDI_UNSUPPORTED_DTYPE, "cubic splines need a float dtype");
    DeviceGuard g(h->device);
    const size_t bytes = (size_t)(h->n - 1) * h->w * elem_size(h->dtype);
    void *na = nullptr, *nb = nullptr; bool oa = false, ob = false;
    ndi_status st = take_table(a, bytes, flags, nullptr, &na, &oa);
    if (st == NDI_OK) st = take_table(b, bytes, flags, nullptr, &nb, &ob);
    if (st == NDI_OK) { cudaError_t e = cudaStreamSynchronize(nullptr); if (e != cudaSuccess) st = cuda_fail(e, "sync"); }
    if (st != NDI_OK) { if (oa) cudaFree(na); if (ob) cudaFree(nb); return st; }
    if (h->owns_coeffs) { cudaFree(h->a); cudaFree(h->b); }
    h->a = na; h->b = nb; h->owns_coeffs = oa;
    h->built_levels = kNotBuilt;
    return NDI_OK;
}

ndi_status ndi_interp1d_cubic_dev(const ndi_interp1d* h, const void* q_dev, int64_t nq, int32_t extrap_mode,
                                  void* out_dev, uint64_t* err_word_dev, void* stream) {
    ndi_status st = check_eval_args(h, q_dev, nq, out_dev); if (st != NDI_OK) return st;
    if (!h->a) return fail(NDI_NO_SPLINE, "no spline coefficients: call ndi_interp1d_spline_build first");
    if (extrap_mode < 0 || extrap_mode > 2) return fail(NDI_INVALID_ARGUMENT, "bad extrapolation mode %d", extrap_mode);
    cudaStream_t s = (cudaStream_t)stream;
    if (err_word_dev) CK(cudaMemsetAsync(err_word_dev, 0xff, sizeof(uint64_t), s));
    return dispatch_float(h->dtype, [&](auto tag) -> ndi_status {
        using T = decltype(tag);
        SearchCfg sc = make_search(h->meta(), h->search_mode, nq, 0);
        return cubic_on_device<T>(h, sc, (const T*)q_dev, nq, extrap_mode, (T*)out_dev, (unsigned long long*)err_word_dev, s);
    });
}

// derivative calls: the argument checks of the value call, then the order (order 0 is ndi_interp1d_cubic itself)
static ndi_status check_cubic_deriv_args(const ndi_interp1d* h, const void* q, int64_t nq, int32_t extrap_mode, int32_t order,
                                         const void* out) {
    ndi_status st = check_eval_args(h, q, nq, out); if (st != NDI_OK) return st;
    if (!h->a) return fail(NDI_NO_SPLINE, "no spline coefficients: call ndi_interp1d_spline_build first");
    if (extrap_mode < 0 || extrap_mode > 2) return fail(NDI_INVALID_ARGUMENT, "bad extrapolation mode %d", extrap_mode);
    if (order != 1 && order != 2) return fail(NDI_INVALID_ARGUMENT, "derivative order must be 1 or 2, got %d", order);
    return NDI_OK;
}

ndi_status ndi_interp1d_cubic_deriv_dev(const ndi_interp1d* h, const void* q_dev, int64_t nq, int32_t extrap_mode, int32_t order,
                                        void* out_dev, uint64_t* err_word_dev, void* stream) {
    ndi_status st = check_cubic_deriv_args(h, q_dev, nq, extrap_mode, order, out_dev); if (st != NDI_OK) return st;
    cudaStream_t s = (cudaStream_t)stream;
    if (err_word_dev) CK(cudaMemsetAsync(err_word_dev, 0xff, sizeof(uint64_t), s));
    return dispatch_float(h->dtype, [&](auto tag) -> ndi_status {
        using T = decltype(tag);
        SearchCfg sc = make_search(h->meta(), h->search_mode, nq, 0);
        return cubic_deriv_on_device<T>(h, sc, (const T*)q_dev, nq, extrap_mode, order, (T*)out_dev, (unsigned long long*)err_word_dev, s);
    });
}

// order 0: the values; 1, 2: the derivatives
static ndi_status cubic_host(const ndi_interp1d* h, const void* q, int64_t nq, int32_t extrap_mode, void* out,
                             uint64_t* word, Phase phase, int64_t nvalid, int32_t order = 0) {
    HostEval he{h->device, elem_size(h->dtype), 1, h->w, {q, nullptr}, nq, out, phase, nvalid};
    return dispatch_float(h->dtype, [&](auto tag) -> ndi_status {
        using T = decltype(tag);
        SearchCfg sc = make_search(h->meta(), h->search_mode, nq, 0);
        const int check = extrap_mode == NDI_EXTRAP_NO ? CHECK_IN_RANGE : (extrap_mode == NDI_EXTRAP_YES ? CHECK_NOT_NAN : CHECK_FINITE_IF_OUTSIDE);
        return run_host_eval(he,
            [&](const void* q0, const void*, int64_t cnt, void* o, unsigned long long* err, cudaStream_t s) -> ndi_status {
                if (order) return cubic_deriv_on_device<T>(h, sc, (const T*)q0, cnt, extrap_mode, order, (T*)o, err, s);
                return cubic_on_device<T>(h, sc, (const T*)q0, cnt, extrap_mode, (T*)o, err, s);
            },
            [&](const void* q0, const void*, int64_t cnt, unsigned long long* err, cudaStream_t s) -> ndi_status {
                CK(launch_validate_queries<T>((const T*)h->x, h->n, nullptr, 0, (const T*)q0, nullptr, cnt, check, err, s));
                return NDI_OK;
            }, word);
    });
}

ndi_status ndi_interp1d_cubic(const ndi_interp1d* h, const void* q, int64_t nq, int32_t extrap_mode, void* out,
                              int64_t* first_bad) {
    if (first_bad) *first_bad = -1;
    ndi_status st = check_eval_args(h, q, nq, out); if (st != NDI_OK) return st;
    if (!h->a) return fail(NDI_NO_SPLINE, "no spline coefficients: call ndi_interp1d_spline_build first");
    if (extrap_mode < 0 || extrap_mode > 2) return fail(NDI_INVALID_ARGUMENT, "bad extrapolation mode %d", extrap_mode);
    uint64_t word;
    if ((st = cubic_host(h, q, nq, extrap_mode, out, &word, Phase::whole, 0)) != NDI_OK) return st;
    return eval1d_status(word, extrap_mode, first_bad);
}

ndi_status ndi_interp1d_cubic_deriv(const ndi_interp1d* h, const void* q, int64_t nq, int32_t extrap_mode, int32_t order,
                                    void* out, int64_t* first_bad) {
    if (first_bad) *first_bad = -1;
    ndi_status st = check_cubic_deriv_args(h, q, nq, extrap_mode, order, out); if (st != NDI_OK) return st;
    uint64_t word;
    if ((st = cubic_host(h, q, nq, extrap_mode, out, &word, Phase::whole, 0, order)) != NDI_OK) return st;
    return eval1d_status(word, extrap_mode, first_bad);
}

// ---- Interp2D ---------------------------------------------------------------------------------------------------
ndi_status ndi_interp2d_create(ndi_dtype dtype, const void* x, int64_t n, const void* y, int64_t m, const void* data,
                               int64_t w, uint32_t flags, ndi_interp2d** out) {
    if (!out) return fail(NDI_INVALID_ARGUMENT, "null handle pointer");
    *out = nullptr;
    if (!dtype_ok(dtype)) return fail(NDI_UNSUPPORTED_DTYPE, "unsupported dtype %d", (int)dtype);
    if (!x || !y || !data) return fail(NDI_INVALID_ARGUMENT, "null pointer");
    if (n < 2 || m < 2 || w < 1) return fail(NDI_INVALID_ARGUMENT, "need n, m >= 2 and w >= 1");
    if (n > 0x7fffffffll || m > 0x7fffffffll) return fail(NDI_INVALID_ARGUMENT, "grid longer than 2^31-1");
    int dev = 0; CK(cudaGetDevice(&dev));
    ndi_status st; Workspace* ws = workspace(dev, &st); if (!ws) return st;
    const size_t es = elem_size(dtype);
    ndi_interp2d* h = new ndi_interp2d();
    h->dtype = dtype; h->device = dev; h->n = n; h->m = m; h->w = w;
    h->x = h->y = h->data = nullptr; h->owns_tables = false;
    h->hint_x = h->hint_y = 0; h->search_mode = NDI_SEARCH_AUTO;
    bool o1 = false, o2 = false, o3 = false;
    st = take_table(x, (size_t)n * es, flags, ws->s[0], &h->x, &o1);
    if (st == NDI_OK) st = take_table(y, (size_t)m * es, flags, ws->s[0], &h->y, &o2);
    if (st == NDI_OK) st = take_table(data, (size_t)n * (size_t)m * (size_t)w * es, flags, ws->s[0], &h->data, &o3);
    if (st != NDI_OK) { if (o1) cudaFree(h->x); if (o2) cudaFree(h->y); if (o3) cudaFree(h->data); delete h; return st; }
    h->owns_tables = o1;
    int32_t rx[2] = {0, 0}, ry[2] = {0, 0};
    st = classify_grid(dtype, h->x, n, ws, rx);
    if (st == NDI_OK) st = classify_grid(dtype, h->y, m, ws, ry);
    if (st == NDI_OK && !(flags & NDI_ASSUME_VALID)) {          // x before y: interp2d/mod.rs:500-509
        if (rx[0] != NDI_MONO_RISING_STRICT) st = fail(NDI_NOT_MONOTONIC, "The x-axis needs to be strictly monotonic rising");
        else if (ry[0] != NDI_MONO_RISING_STRICT) st = fail(NDI_NOT_MONOTONIC, "The y-axis needs to be strictly monotonic rising");
    }
    if (st != NDI_OK) { ndi_interp2d_destroy(h); return st; }
    h->hint_x = rx[0] == NDI_MONO_RISING_STRICT ? rx[1] : 0;
    h->hint_y = ry[0] == NDI_MONO_RISING_STRICT ? ry[1] : 0;
    if (!h->hint_x) st = build_aids(dtype, h->x, n, ws->s[0], &h->aids_x);
    if (st == NDI_OK && !h->hint_y) st = build_aids(dtype, h->y, m, ws->s[0], &h->aids_y);
    if (st == NDI_OK) st = scan_fast_tables(dtype, h->data, (size_t)n * (size_t)m * (size_t)w, ws, &h->fast_tables);
    if (st != NDI_OK) { ndi_interp2d_destroy(h); return st; }
    *out = h;
    return NDI_OK;
}

ndi_status ndi_interp2d_create_strided(ndi_dtype dtype, const void* x, int64_t n, int64_t x_stride, const void* y,
                                       int64_t m, int64_t y_stride, const void* data, int32_t ndim, const int64_t* shape,
                                       const int64_t* strides, uint32_t flags, ndi_interp2d** out) {
    if (!out) return fail(NDI_INVALID_ARGUMENT, "null handle pointer");
    *out = nullptr;
    if (!dtype_ok(dtype)) return fail(NDI_UNSUPPORTED_DTYPE, "unsupported dtype %d", (int)dtype);
    if (!x || !y || !data || !shape || !strides) return fail(NDI_INVALID_ARGUMENT, "null pointer");
    if (flags & NDI_BORROW) return fail(NDI_INVALID_ARGUMENT, "a strided view cannot be borrowed: the kernels read dense tables");
    if (ndim < 2 || ndim > kMaxDims) return fail(NDI_INVALID_ARGUMENT, "data needs 2..%d dimensions", kMaxDims);
    if (shape[0] != n || shape[1] != m)
        return fail(NDI_INVALID_ARGUMENT, "data.shape[0..2] = (%lld, %lld) but the axes have (%lld, %lld) elements",
                    (long long)shape[0], (long long)shape[1], (long long)n, (long long)m);
    int dev = 0; CK(cudaGetDevice(&dev));
    ndi_status st; Workspace* ws = workspace(dev, &st); if (!ws) return st;
    const size_t es = elem_size(dtype);
    const bool dsrc = (flags & NDI_DEVICE_POINTERS) != 0;
    int64_t w = 1;
    for (int k = 2; k < ndim; ++k) w *= shape[k];
    void *xd = nullptr, *yd = nullptr, *dd = nullptr;
    st = pack_view(x, es, 1, &n, &x_stride, dsrc, ws->s[0], &xd);
    if (st == NDI_OK) st = pack_view(y, es, 1, &m, &y_stride, dsrc, ws->s[0], &yd);
    if (st == NDI_OK) st = pack_view(data, es, ndim, shape, strides, dsrc, ws->s[0], &dd);
    if (st == NDI_OK) st = ndi_interp2d_create(dtype, xd, n, yd, m, dd, w, (flags & NDI_ASSUME_VALID) | NDI_DEVICE_POINTERS | NDI_BORROW, out);
    if (st != NDI_OK) { cudaFree(xd); cudaFree(yd); cudaFree(dd); return st; }
    (*out)->owns_tables = true;
    return NDI_OK;
}

ndi_status ndi_interp2d_destroy(ndi_interp2d* h) {
    if (!h) return NDI_OK;
    DeviceGuard g(h->device);
    if (h->owns_tables) { cudaFree(h->x); cudaFree(h->y); cudaFree(h->data); }
    h->aids_x.release(); h->aids_y.release();
    delete h;
    return NDI_OK;
}
ndi_status ndi_interp2d_info(const ndi_interp2d* h, ndi_dtype* dtype, int64_t* n, int64_t* m, int64_t* w, int32_t* device) {
    if (!h) return fail(NDI_INVALID_ARGUMENT, "null handle");
    if (dtype) *dtype = h->dtype;
    if (n) *n = h->n;
    if (m) *m = h->m;
    if (w) *w = h->w;
    if (device) *device = h->device;
    return NDI_OK;
}
ndi_status ndi_interp2d_set_search_mode(ndi_interp2d* h, int32_t mode) {
    if (!h || mode < 0 || mode > NDI_SEARCH_MERGE) return fail(NDI_INVALID_ARGUMENT, "bad search mode");
    h->search_mode = mode;
    return NDI_OK;
}
ndi_status ndi_interp2d_device_ptrs(const ndi_interp2d* h, const void** x, const void** y, const void** data) {
    if (!h) return fail(NDI_INVALID_ARGUMENT, "null handle");
    if (x) *x = h->x;
    if (y) *y = h->y;
    if (data) *data = h->data;
    return NDI_OK;
}
ndi_status ndi_interp2d_clone_to_device(const ndi_interp2d* h, int32_t device, ndi_interp2d** out) {
    return clone_to_device(h, device, out, ndi_interp2d_destroy, [&](ndi_interp2d* c, auto& copy) {
        const size_t es = elem_size(h->dtype);
        c->owns_tables = true;
        c->x = c->y = c->data = nullptr;
        c->aids_x = c->aids_y = GridAids{};
        ndi_status st = copy(&c->x, h->x, (size_t)h->n * es);
        if (st == NDI_OK) st = copy(&c->y, h->y, (size_t)h->m * es);
        if (st == NDI_OK) st = copy(&c->data, h->data, (size_t)h->n * h->m * h->w * es);
        if (st == NDI_OK && !h->hint_x) st = build_aids(c->dtype, c->x, c->n, nullptr, &c->aids_x);
        if (st == NDI_OK && !h->hint_y) st = build_aids(c->dtype, c->y, c->m, nullptr, &c->aids_y);
        return st;
    });
}

static void search2(const ndi_interp2d* h, size_t es, int64_t nq, SearchCfg* sx, SearchCfg* sy) {
    *sx = make_search(h->meta_x(), h->search_mode, nq, 0);
    *sy = make_search(h->meta_y(), h->search_mode, nq, sx->smem ? (size_t)sx->stage_n * es + 16 : 0);
}

ndi_status ndi_interp2d_set_binning(ndi_interp2d* h, int32_t mode, int32_t band_rows) {
    if (!h || mode < NDI_BIN_AUTO || mode > NDI_BIN_SWEEP || band_rows < 0) return fail(NDI_INVALID_ARGUMENT, "bad binning mode");
    h->bin_mode = mode; h->band_rows = band_rows;
    return NDI_OK;
}

}  // extern "C"

namespace {

// Is grouping the queries by table band (ndi_bin.cu) worth its two extra passes?  Measured on B200
// (profiles/r01/binning.md): yes when the table cannot stay in L2 under random gathers AND an
// output row is at least two sectors (C5a, 128-byte rows: 3.44 -> 2.54 ms); no for 32-byte rows
// (C4: 0.59 -> 0.62 ms), where the scattered output stores and the binning passes cost what the
// gathers save and the evaluation is bound by L1 wavefronts either way.
bool want_binning(const ndi_interp2d* h, int64_t nq, size_t es, BandPlan* bp) {
    constexpr size_t kBandBytes = 16ull << 20;
    if (h->bin_mode == NDI_BIN_OFF || h->bin_mode == NDI_BIN_SWEEP || nq < 2 || nq > 0xffffffffll) return false;
    const double table = (double)h->n * (double)h->m * (double)h->w * (double)es;
    *bp = plan_bands(h->n, h->m, h->w, es, kBandBytes, h->band_rows);
    if (bp->nbands < 2) return false;
    if (h->bin_mode == NDI_BIN_ON) return true;
    const double resident = 0.4 * (double)device_info().l2_bytes;   // what random gathers keep of L2 (two partitions, output stream)
    const double seg = (double)(h->w * es);
    if (table <= resident || nq < (1 << 18) || seg < 64) return false;
    const double direct = (double)nq * 4.0 * seg * (1.0 - resident / table);
    const double binned = table + (double)nq * (double)(es + 2 * (4 + 2 * es));
    return direct > 1.5 * binned;
}

// Band sweeps (ndi_sweep.cu): the batch stays where it is and is walked once per table band.  Built for thin rows on a
// table a few times the size of L2 (C4: 134 MB, four sweeps of 32 MB).  MEASURED, AND NOT CHOSEN BY AUTO: the sweeps cut
// C4's DRAM traffic from 3.14 to 1.36 GB as designed, but the compaction, the scattered 32-byte output rows and the lower
// occupancy cost more than the DRAM time they save -- 0.580 ms against 0.537 ms for the direct kernel, which already runs
// at the DRAM ceiling of its access pattern (profiles/r02/sweeps_and_probes.md).  The mode stays selectable
// (NDI_BIN_SWEEP through ndi_interp2d_set_binning) and is covered by the parity tests.
bool want_sweeps(const ndi_interp2d* h, int64_t nq, size_t es, const void* out, SweepPlan* sp) {
    constexpr size_t kSweepBandBytes = 32ull << 20;
    if (h->bin_mode != NDI_BIN_SWEEP) return false;
    if (!sweep_shape_ok(h->n, h->m, h->w, es, h->data, out, nq)) return false;
    *sp = plan_sweeps(h->n, h->m, h->w, es, kSweepBandBytes, h->band_rows);
    return true;
}

// one bilinear evaluation of a device-resident batch: direct, in band sweeps, or binned by table band
template <class T>
ndi_status bilinear_on_device(const ndi_interp2d* h, const SearchCfg& sx, const SearchCfg& sy, const T* qx, const T* qy,
                              int64_t nq, int extrapolate, T* out, unsigned long long* err, cudaStream_t s) {
    SweepPlan sp;
    if (want_sweeps(h, nq, sizeof(T), out, &sp)) {
        unsigned long long* ticket = nullptr;
        CK(cudaMallocAsync((void**)&ticket, sizeof(unsigned long long), s));
        cudaError_t e = cudaMemsetAsync(ticket, 0, sizeof(unsigned long long), s);
        if (e == cudaSuccess)
            e = launch_interp2d_bilinear_sweep<T>((const T*)h->x, h->n, sx, (const T*)h->y, h->m, sy, (const T*)h->data, h->w, qx, qy,
                                                  nq, extrapolate, out, err, h->fast_tables, sp, ticket, s);
        cudaFreeAsync(ticket, s);
        if (e != cudaSuccess) return cuda_fail(e, "swept bilinear launch");
        return NDI_OK;
    }
    BandPlan bp;
    if (!want_binning(h, nq, sizeof(T), &bp)) {
        CK(launch_interp2d_bilinear<T>((const T*)h->x, h->n, sx, (const T*)h->y, h->m, sy, (const T*)h->data, h->w, qx, qy, nq,
                                       extrapolate, out, err, nullptr, h->fast_tables, nullptr, s));
        return NDI_OK;
    }
    void* scratch = nullptr;
    CK(cudaMallocAsync(&scratch, bin_scratch_bytes(nq, sizeof(T)), s));
    // the scatter kernel keeps its chunk in static shared memory: leave room when staging the grid
    const SearchCfg sbin = make_search(h->meta_x(), h->search_mode, nq, 48 * 1024);
    const unsigned* perm = nullptr; const T *bx = nullptr, *by = nullptr;
    unsigned long long* next_task = nullptr;
    cudaError_t e = launch_bin_queries<T>((const T*)h->x, h->n, sbin, qx, qy, nq, bp, scratch, &perm, &bx, &by, &next_task, s);
    if (e == cudaSuccess)
        e = launch_interp2d_bilinear<T>((const T*)h->x, h->n, sx, (const T*)h->y, h->m, sy, (const T*)h->data, h->w, bx, by, nq,
                                        extrapolate, out, err, perm, h->fast_tables, next_task, s);
    cudaFreeAsync(scratch, s);
    if (e != cudaSuccess) return cuda_fail(e, "binned bilinear launch");
    return NDI_OK;
}

}  // namespace

extern "C" {

ndi_status ndi_interp2d_bilinear_dev(const ndi_interp2d* h, const void* qx_dev, const void* qy_dev, int64_t nq,
                                     int32_t extrapolate, void* out_dev, uint64_t* err_word_dev, void* stream) {
    ndi_status st = check_eval_args(h, qx_dev, nq, out_dev); if (st != NDI_OK) return st;
    if (nq > 0 && !qy_dev) return fail(NDI_INVALID_ARGUMENT, "null pointer");
    cudaStream_t s = (cudaStream_t)stream;
    if (err_word_dev) CK(cudaMemsetAsync(err_word_dev, 0xff, sizeof(uint64_t), s));
    return dispatch(h->dtype, [&](auto tag) -> ndi_status {
        using T = decltype(tag);
        SearchCfg sx, sy; search2(h, sizeof(T), nq, &sx, &sy);
        return bilinear_on_device<T>(h, sx, sy, (const T*)qx_dev, (const T*)qy_dev, nq, extrapolate != 0, (T*)out_dev,
                                     (unsigned long long*)err_word_dev, s);
    });
}

static ndi_status bilinear_host(const ndi_interp2d* h, const void* qx, const void* qy, int64_t nq, int32_t extrapolate,
                                void* out, uint64_t* word, Phase phase, int64_t nvalid) {
    HostEval he{h->device, elem_size(h->dtype), 2, h->w, {qx, qy}, nq, out, phase, nvalid};
    return dispatch(h->dtype, [&](auto tag) -> ndi_status {
        using T = decltype(tag);
        SearchCfg sx, sy; search2(h, sizeof(T), nq, &sx, &sy);
        return run_host_eval(he,
            [&](const void* q0, const void* q1, int64_t cnt, void* o, unsigned long long* err, cudaStream_t s) -> ndi_status {
                return bilinear_on_device<T>(h, sx, sy, (const T*)q0, (const T*)q1, cnt, extrapolate != 0, (T*)o, err, s);
            },
            [&](const void* q0, const void* q1, int64_t cnt, unsigned long long* err, cudaStream_t s) -> ndi_status {
                CK(launch_validate_queries<T>((const T*)h->x, h->n, (const T*)h->y, h->m, (const T*)q0, (const T*)q1, cnt,
                                              extrapolate ? CHECK_NOT_NAN : CHECK_IN_RANGE, err, s));
                return NDI_OK;
            }, word);
    });
}
static ndi_status eval2d_status(uint64_t word, int nan_only, int64_t* first_bad, int32_t* bad_axis) {
    if (word == NDI_ERR_WORD_NONE) return NDI_OK;
    const int64_t idx = (int64_t)(word >> 1);
    const int axis = (int)(word & 1);
    if (first_bad) *first_bad = idx;
    if (bad_axis) *bad_axis = axis;
    return nan_only ? fail(NDI_NAN_QUERY, "not implemented: failed to convert NaN to usize (query %lld)", (long long)idx)
                    : fail(NDI_OUT_OF_BOUNDS, "%s of query %lld is not in range", axis ? "y" : "x", (long long)idx);
}

ndi_status ndi_interp2d_bilinear(const ndi_interp2d* h, const void* qx, const void* qy, int64_t nq, int32_t extrapolate,
                                 void* out, int64_t* first_bad, int32_t* bad_axis) {
    if (first_bad) *first_bad = -1;
    if (bad_axis) *bad_axis = -1;
    ndi_status st = check_eval_args(h, qx, nq, out); if (st != NDI_OK) return st;
    if (nq > 0 && !qy) return fail(NDI_INVALID_ARGUMENT, "null pointer");
    uint64_t word;
    if ((st = bilinear_host(h, qx, qy, nq, extrapolate, out, &word, Phase::whole, 0)) != NDI_OK) return st;
    return eval2d_status(word, extrapolate, first_bad, bad_axis);
}

}  // extern "C"

// ---- one interpolator on several devices of this process (SURVEY.md section 8(b): ndi_replicate) ------------------
// The tables are peer-copied to every device (ndi_interp*_clone_to_device); a host call cuts the batch into
// contiguous blocks of queries, one per device (SURVEY.md section 8(e): keeps sorted batches sorted and makes the
// first failing query a minimum over the blocks), and runs the blocks concurrently, each on its own worker thread
// with its own per-thread workspace (streams, pinned staging).  No collective, no data shared between the blocks.
namespace {

class Workers {                                   // one persistent thread per device of a group
public:
    explicit Workers(int n) : slots_(n) {
        for (int i = 0; i < n; ++i) threads_.emplace_back([this, i] { run(i); });
    }
    ~Workers() {
        { std::lock_guard<std::mutex> lk(mu_); stop_ = true; }
        cv_.notify_all();
        for (auto& t : threads_) t.join();
    }
    // fn(member) on every worker; returns the first non-OK status (and its message, into this thread's slot)
    ndi_status all(const std::function<ndi_status(int)>& fn) {
        std::unique_lock<std::mutex> lk(mu_);
        fn_ = &fn; pending_ = (int)slots_.size(); ++epoch_;
        for (auto& s : slots_) { s.todo = true; s.st = NDI_OK; }
        cv_.notify_all();
        done_.wait(lk, [&] { return pending_ == 0; });
        for (auto& s : slots_)
            if (s.st != NDI_OK) { snprintf(g_err, sizeof(g_err), "%s", s.msg); return s.st; }
        return NDI_OK;
    }
private:
    struct Slot { bool todo = false; ndi_status st = NDI_OK; char msg[512] = ""; };
    void run(int i) {
        for (;;) {
            const std::function<ndi_status(int)>* fn;
            {
                std::unique_lock<std::mutex> lk(mu_);
                cv_.wait(lk, [&] { return stop_ || slots_[i].todo; });
                if (stop_) return;
                slots_[i].todo = false;
                fn = fn_;
            }
            const ndi_status st = (*fn)(i);
            std::lock_guard<std::mutex> lk(mu_);
            slots_[i].st = st;
            if (st != NDI_OK) snprintf(slots_[i].msg, sizeof(slots_[i].msg), "%s", g_err);
            if (--pending_ == 0) done_.notify_all();
        }
    }
    std::mutex mu_; std::condition_variable cv_, done_;
    std::vector<Slot> slots_; std::vector<std::thread> threads_;
    const std::function<ndi_status(int)>* fn_ = nullptr; int pending_ = 0; unsigned long long epoch_ = 0; bool stop_ = false;
};

// block k of nq queries cut into nd contiguous blocks whose starts are multiples of 32
inline int64_t block_start(int64_t nq, int nd, int k) { return k >= nd ? nq : ((nq * k / nd) & ~31ll); }

constexpr int64_t kGroupMinQueries = 1 << 15;       // below this a batch stays on the first device (latency path)

}  // namespace

// the C ABI's ndi_interp1d_group and ndi_interp2d_group: members[k] lives on the k-th device of the group
template <class H>
struct Group {
    std::vector<H*> members; std::vector<char> owned;   // owned: a clone, destroyed with the group
    Workers pool;
    ndi_status (*destroy)(H*);
    Group(int n, ndi_status (*destroy_handle)(H*)) : pool(n), destroy(destroy_handle) {}
    ~Group() { for (size_t k = 0; k < members.size(); ++k) if (owned[k]) destroy(members[k]); }
};
struct ndi_interp1d_group : Group<ndi_interp1d> { using Group::Group; };
struct ndi_interp2d_group : Group<ndi_interp2d> { using Group::Group; };

namespace {

template <class G, class H>
ndi_status replicate(const H* h, const int32_t* devices, int32_t ndev, G** out, ndi_status (*clone)(const H*, int32_t, H**),
                     ndi_status (*destroy)(H*)) {
    if (!h || !devices || !out || ndev < 1 || ndev > 64) return fail(NDI_INVALID_ARGUMENT, "need a handle and 1..64 devices");
    *out = nullptr;
    int count = 0; CK(cudaGetDeviceCount(&count));
    for (int k = 0; k < ndev; ++k) {
        if (devices[k] < 0 || devices[k] >= count) return fail(NDI_INVALID_ARGUMENT, "device %d does not exist (%d visible)", devices[k], count);
        for (int j = 0; j < k; ++j) if (devices[j] == devices[k]) return fail(NDI_INVALID_ARGUMENT, "device %d listed twice", devices[k]);
    }
    G* g = new G(ndev, destroy);
    for (int k = 0; k < ndev; ++k) {
        if (devices[k] == h->device) { g->members.push_back(const_cast<H*>(h)); g->owned.push_back(0); continue; }
        H* c = nullptr;
        const ndi_status st = clone(h, devices[k], &c);
        if (st != NDI_OK) { delete g; return st; }
        g->members.push_back(c); g->owned.push_back(1);
    }
    *out = g;
    return NDI_OK;
}

// One host call on a group.  A batch below kGroupMinQueries, or on a group of one device, is single(first member).
// A larger one is checked by check(first member) and fanned out in two phases: block(member, lo, cnt, phase, nvalid,
// &word) runs the block of queries [lo, lo + cnt) on its member's worker thread, first Phase::prepass on every block,
// then Phase::evaluate on the rows before the batch-wide first failure.  status(word) turns that failure's error
// word into the call's status.
template <class H, class Single, class Check, class Block, class Status>
ndi_status group_call(Group<H>* g, int64_t nq, int ncoord, Single&& single, Check&& check, Block&& block, Status&& status) {
    if (!g || g->members.empty()) return fail(NDI_INVALID_ARGUMENT, "null group");
    const int nd = (int)g->members.size();
    if (nd == 1 || nq < kGroupMinQueries) return single(g->members[0]);
    ndi_status st = check(g->members[0]); if (st != NDI_OK) return st;
    std::vector<uint64_t> words((size_t)nd, NDI_ERR_WORD_NONE);
    st = g->pool.all([&](int k) -> ndi_status {
        const int64_t lo = block_start(nq, nd, k), cnt = block_start(nq, nd, k + 1) - lo;
        return cnt > 0 ? block(g->members[(size_t)k], lo, cnt, Phase::prepass, 0, &words[(size_t)k]) : NDI_OK;
    });
    if (st != NDI_OK) return st;
    uint64_t word = NDI_ERR_WORD_NONE;
    for (int k = 0; k < nd; ++k) {
        if (words[(size_t)k] == NDI_ERR_WORD_NONE) continue;
        const uint64_t w = err_rebase(words[(size_t)k], ncoord, block_start(nq, nd, k));
        if (w < word) word = w;
    }
    const int64_t first = word == NDI_ERR_WORD_NONE ? nq : err_query(word, ncoord);   // rows before `first` are evaluated
    st = g->pool.all([&](int k) -> ndi_status {
        const int64_t lo = block_start(nq, nd, k), cnt = block_start(nq, nd, k + 1) - lo;
        const int64_t nvalid = first - lo < cnt ? first - lo : cnt;
        uint64_t unused;
        return (cnt > 0 && nvalid > 0) ? block(g->members[(size_t)k], lo, cnt, Phase::evaluate, nvalid, &unused) : NDI_OK;
    });
    return st != NDI_OK ? st : status(word);
}

}  // namespace

extern "C" {

ndi_status ndi_interp1d_replicate(const ndi_interp1d* h, const int32_t* devices, int32_t ndev, ndi_interp1d_group** out) {
    return replicate(h, devices, ndev, out, ndi_interp1d_clone_to_device, ndi_interp1d_destroy);
}
ndi_status ndi_interp1d_group_destroy(ndi_interp1d_group* g) {
    delete g;
    return NDI_OK;
}
ndi_status ndi_interp1d_group_size(const ndi_interp1d_group* g, int32_t* ndev) {
    if (!g || !ndev) return fail(NDI_INVALID_ARGUMENT, "null pointer");
    *ndev = (int32_t)g->members.size();
    return NDI_OK;
}

ndi_status ndi_interp1d_group_linear(ndi_interp1d_group* g, const void* q, int64_t nq, int32_t extrapolate, void* out,
                                     int64_t* first_bad) {
    if (first_bad) *first_bad = -1;
    return group_call(g, nq, 1,
        [&](const ndi_interp1d* h0) { return ndi_interp1d_linear(h0, q, nq, extrapolate, out, first_bad); },
        [&](const ndi_interp1d* h0) { return check_eval_args(h0, q, nq, out); },
        [&](const ndi_interp1d* h, int64_t lo, int64_t cnt, Phase phase, int64_t nvalid, uint64_t* w) {
            const size_t es = elem_size(h->dtype);
            return linear_host(h, (const unsigned char*)q + (size_t)lo * es, cnt, extrapolate,
                               (unsigned char*)out + (size_t)lo * h->w * es, w, phase, nvalid);
        },
        [&](uint64_t word) { return eval1d_status(word, extrapolate, first_bad); });
}

ndi_status ndi_interp1d_group_cubic(ndi_interp1d_group* g, const void* q, int64_t nq, int32_t extrap_mode, void* out,
                                    int64_t* first_bad) {
    if (first_bad) *first_bad = -1;
    return group_call(g, nq, 1,
        [&](const ndi_interp1d* h0) { return ndi_interp1d_cubic(h0, q, nq, extrap_mode, out, first_bad); },
        [&](const ndi_interp1d* h0) {
            ndi_status st = check_eval_args(h0, q, nq, out); if (st != NDI_OK) return st;
            if (!h0->a) return fail(NDI_NO_SPLINE, "no spline coefficients: build the spline before ndi_interp1d_replicate");
            if (extrap_mode < 0 || extrap_mode > 2) return fail(NDI_INVALID_ARGUMENT, "bad extrapolation mode %d", extrap_mode);
            return NDI_OK;
        },
        [&](const ndi_interp1d* h, int64_t lo, int64_t cnt, Phase phase, int64_t nvalid, uint64_t* w) {
            const size_t es = elem_size(h->dtype);
            return cubic_host(h, (const unsigned char*)q + (size_t)lo * es, cnt, extrap_mode,
                              (unsigned char*)out + (size_t)lo * h->w * es, w, phase, nvalid);
        },
        [&](uint64_t word) { return eval1d_status(word, extrap_mode, first_bad); });
}

ndi_status ndi_interp1d_group_linear_deriv(ndi_interp1d_group* g, const void* q, int64_t nq, int32_t extrapolate, void* out,
                                           int64_t* first_bad) {
    if (first_bad) *first_bad = -1;
    return group_call(g, nq, 1,
        [&](const ndi_interp1d* h0) { return ndi_interp1d_linear_deriv(h0, q, nq, extrapolate, out, first_bad); },
        [&](const ndi_interp1d* h0) { return check_eval_args(h0, q, nq, out); },
        [&](const ndi_interp1d* h, int64_t lo, int64_t cnt, Phase phase, int64_t nvalid, uint64_t* w) {
            const size_t es = elem_size(h->dtype);
            return linear_host(h, (const unsigned char*)q + (size_t)lo * es, cnt, extrapolate,
                               (unsigned char*)out + (size_t)lo * h->w * es, w, phase, nvalid, true);
        },
        [&](uint64_t word) { return eval1d_status(word, extrapolate, first_bad); });
}

ndi_status ndi_interp1d_group_cubic_deriv(ndi_interp1d_group* g, const void* q, int64_t nq, int32_t extrap_mode, int32_t order,
                                          void* out, int64_t* first_bad) {
    if (first_bad) *first_bad = -1;
    return group_call(g, nq, 1,
        [&](const ndi_interp1d* h0) { return ndi_interp1d_cubic_deriv(h0, q, nq, extrap_mode, order, out, first_bad); },
        [&](const ndi_interp1d* h0) { return check_cubic_deriv_args(h0, q, nq, extrap_mode, order, out); },
        [&](const ndi_interp1d* h, int64_t lo, int64_t cnt, Phase phase, int64_t nvalid, uint64_t* w) {
            const size_t es = elem_size(h->dtype);
            return cubic_host(h, (const unsigned char*)q + (size_t)lo * es, cnt, extrap_mode,
                              (unsigned char*)out + (size_t)lo * h->w * es, w, phase, nvalid, order);
        },
        [&](uint64_t word) { return eval1d_status(word, extrap_mode, first_bad); });
}

ndi_status ndi_interp2d_replicate(const ndi_interp2d* h, const int32_t* devices, int32_t ndev, ndi_interp2d_group** out) {
    return replicate(h, devices, ndev, out, ndi_interp2d_clone_to_device, ndi_interp2d_destroy);
}
ndi_status ndi_interp2d_group_destroy(ndi_interp2d_group* g) {
    delete g;
    return NDI_OK;
}

ndi_status ndi_interp2d_group_bilinear(ndi_interp2d_group* g, const void* qx, const void* qy, int64_t nq, int32_t extrapolate,
                                       void* out, int64_t* first_bad, int32_t* bad_axis) {
    if (first_bad) *first_bad = -1;
    if (bad_axis) *bad_axis = -1;
    return group_call(g, nq, 2,
        [&](const ndi_interp2d* h0) { return ndi_interp2d_bilinear(h0, qx, qy, nq, extrapolate, out, first_bad, bad_axis); },
        [&](const ndi_interp2d* h0) {
            ndi_status st = check_eval_args(h0, qx, nq, out); if (st != NDI_OK) return st;
            return qy ? NDI_OK : fail(NDI_INVALID_ARGUMENT, "null pointer");
        },
        [&](const ndi_interp2d* h, int64_t lo, int64_t cnt, Phase phase, int64_t nvalid, uint64_t* w) {
            const size_t es = elem_size(h->dtype);
            return bilinear_host(h, (const unsigned char*)qx + (size_t)lo * es, (const unsigned char*)qy + (size_t)lo * es, cnt,
                                 extrapolate, (unsigned char*)out + (size_t)lo * h->w * es, w, phase, nvalid);
        },
        [&](uint64_t word) { return eval2d_status(word, extrapolate, first_bad, bad_axis); });
}

}  // extern "C"
