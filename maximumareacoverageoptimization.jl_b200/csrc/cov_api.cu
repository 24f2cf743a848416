// cov_api.cu -- the C ABI of libcoverage_cuda (include/coverage_cuda.h): handle lifecycle, the
// device-resident cell store, parameter upload, and the batched evaluation pipelines.
//
// The reference (/root/reference, pure Julia) has no FFI; each entry point replaces the Julia
// lines cited beside its declaration in include/coverage_cuda.h. Nothing here computes coverage
// on the CPU: without a CUDA device every entry point that needs one fails with COV_ERR_CUDA.
#include <cuda_runtime.h>
#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdlib>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <string>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <thread>
#include <unordered_map>
#include <vector>
#include "cov_device.cuh"
#include "cov_kernels.cuh"
#include "cov_region.cuh"
#include "../../include/coverage_cuda.h"

using namespace cov;


// ------------------------------------------------------------------------------------------
// a few host threads for the staging copies of pageable buffers (a Julia Array is pageable: one
// thread's memcpy into the pinned staging buffer would cap the host path at ~10 GB/s)
// ------------------------------------------------------------------------------------------
class CopyPool {
public:
    explicit CopyPool(int n)
    {
        for (int k = 0; k < n; ++k) workers_.emplace_back([this] { run(); });
    }
    ~CopyPool()
    {
        {
            std::lock_guard<std::mutex> lk(m_);
            stop_.store(true);
        }
        cv_.notify_all();
        for (auto &t : workers_) t.join();
    }
    // memcpy split over the pool and the calling thread; returns when all of it is done
    void copy(void *dst, const void *src, size_t bytes)
    {
        const size_t parts = workers_.size() + 1;
        if (bytes < (1u << 20) || parts == 1) {
            memcpy(dst, src, bytes);
            return;
        }
        const size_t per = ((bytes + parts - 1) / parts + 4095) / 4096 * 4096;
        int posted = 0;
        {
            std::lock_guard<std::mutex> lk(m_);
            for (size_t k = 1; k < parts; ++k) {
                const size_t off = k * per;
                if (off >= bytes) break;
                const size_t n = std::min(per, bytes - off);
                tasks_.push_back([=] { memcpy((char *)dst + off, (const char *)src + off, n); });
                ++posted;
            }
            pending_.fetch_add(posted);
            avail_.fetch_add(posted);
        }
        cv_.notify_all();
        memcpy(dst, src, std::min(per, bytes));
        // the parts are short (a few hundred microseconds at most): wait for them without sleeping
        for (unsigned spins = 0; pending_.load(std::memory_order_acquire) != 0; ++spins) {
            if ((spins & 1023u) == 1023u) std::this_thread::yield();
            else relax();
        }
    }

private:
    static void relax()
    {
#if defined(__x86_64__) || defined(__i386__)
        __builtin_ia32_pause();
#else
        std::this_thread::yield();
#endif
    }
    // Workers stay awake for about a millisecond after their last job: the slices of one pipelined call arrive
    // every few hundred microseconds, and a futex wake-up per slice cost more than the copy itself.
    void run()
    {
        for (;;) {
            const auto idle_since = std::chrono::steady_clock::now();
            unsigned spins = 0;
            while (avail_.load(std::memory_order_acquire) == 0 && !stop_.load(std::memory_order_relaxed)) {
                relax();
                if ((++spins & 255u) == 0 &&
                    std::chrono::steady_clock::now() - idle_since > std::chrono::microseconds(1000)) {
                    std::unique_lock<std::mutex> lk(m_);
                    cv_.wait(lk, [this] { return stop_.load() || avail_.load() > 0; });
                    break;
                }
            }
            std::function<void()> job;
            {
                std::lock_guard<std::mutex> lk(m_);
                if (tasks_.empty()) {
                    if (stop_.load()) return;
                    continue;
                }
                job = std::move(tasks_.back());
                tasks_.pop_back();
                avail_.fetch_sub(1);
            }
            job();
            pending_.fetch_sub(1, std::memory_order_release);
        }
    }
    std::vector<std::thread> workers_;
    std::vector<std::function<void()>> tasks_;
    std::mutex m_;
    std::condition_variable cv_;
    std::atomic<int> pending_{0}, avail_{0};
    std::atomic<bool> stop_{false};
};

// ------------------------------------------------------------------------------------------
// handle
// ------------------------------------------------------------------------------------------
struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
};

// Pinned host scratch for the few words a call brings back or sends (one field per use, allocated once per handle).
struct HostScratch {
    unsigned long long stats[2 + kMaxClasses]; // rebuild_planes: entries, cells, per-class OR of the multiplicities
    int overflow;                              // upload_points, cov_fire_step
    unsigned long long removed;                // cov_remove_covered, cov_fire_step: entries removed / pushed
    double fire_p[9];                          // cov_fire_step: direction probabilities
    double win_obj;                            // the poll winner of one device window (enqueue_winner)
    long long win_idx;
    int region_arcs;                           // cov_set_region
};
// h_poll, the pinned scratch of the small-batch path: candidates at 0 (<= 256 KiB), results from kPollOut on
constexpr size_t kPollBytes = 2u << 20, kPollOut = 512u << 10;

struct cov_handle {
    int device = 0;
    cudaStream_t own_stream = nullptr, stream = nullptr; // stream = own_stream or an adopted one
    cudaStream_t s_in = nullptr, s_out = nullptr;        // copy engines of the host pipeline
    std::string err;

    // cell store
    bool have_grid = false;
    DevBuf mult, cls, planes, planes_q;
    GridDesc g{};
    int64_t n_entries = 0, n_cells = 0;
    int area_exact = 0;
    // The point list in the reference's order, for the ordered kernel (area_exact == 0 or COV_KERNEL_ORDERED).
    // ent_known: the host mirror follows the order cov_set_points / cov_add_points gave (removals pending in
    // ent_removed_pending are applied lazily: every entry of a covered cell goes, the others keep their order);
    // otherwise the order is createPOI's (i outer, j inner, duplicates together), built from the cell store on demand.
    // The first cov_add_points on such a store builds the mirror in that order and appends to it.
    std::vector<int> ent_cell_h;
    std::vector<unsigned char> ent_cls_h;
    bool ent_known = false, ent_removed_pending = false, ent_dev_valid = false;
    DevBuf ent_cell, ent_cls;

    // closure parameters
    bool have_params = false;
    ObjParams o{};
    DevBuf params; // 5N doubles: r_max, prev_x, prev_y, prev_z, cons3_G

    // the grid-free static objective (cov_set_region): domain, covered discs, the arcs of their boundary
    bool have_region = false;
    RegionDesc region{};
    DevBuf region_discs, region_arcs, region_count, d_area;

    LaunchCfg cfg{};
    int64_t chunk = 0;

    // scratch
    DevBuf counter, stats, xyT, small_in, argmin_obj, argmin_idx, removed, overflow;
    DevBuf backup; // mult + cls before an append, restored when the append fails (overflow, mixed weights)
    // forest-fire automaton state (ping-pong) and its direction probabilities
    DevBuf fire[2], fire_p;
    int fire_cur = 0;
    bool have_fire = false;
    // evaluation window (device) and staging (pinned host)
    DevBuf dX, d_obj, d_count, d_feas, d_clscnt, d_prog;
    DevBuf d_raw[2]; // packed slices as they arrive (cov_eval_batch_packed), widened into dX
    DevBuf mads_in, mads_out; // cov_mads_solve_batch: starts, initial meshes, powers of ten / results
    DevBuf ens;               // cov_run_horizon_ensemble: the scenarios' stores, plane sets, parameters and thresholds
                              // (E times the store: freed when the call ends, never kept between calls)
    void *h_in[2] = {nullptr, nullptr};
    size_t h_in_cap = 0;
    void *h_out = nullptr;
    size_t h_out_cap = 0;
    HostScratch *h_small = nullptr;
    void *h_poll = nullptr; // pinned scratch of the small-batch path (kPollBytes)
    size_t h_poll_cap = 0;

    std::vector<cudaEvent_t> ev_pool; // recycled
    // (start, stop) events around every coverage-kernel launch since the last drain
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> kernel_spans;
    size_t last_call_begin = 0;   // first span of the last eval call
    double drained_ms = 0;        // spans already folded into the running total
    int64_t drained_launches = 0;
    double last_call_ms_cache = -1;
    int64_t launches = 0;
    LaunchInfo last_info{};
    int counter_next = 0; // next unused slot of the zeroed counter ring
    CopyPool *pool = nullptr; // created on the first large pageable transfer
    // COV_OPT_TRACE: per-slice timeline of the last host-path call (ms since its first copy was queued)
    int trace = 0;
    int zero_copy_out = 1; // COV_OPT_ZEROCOPY_OUT: kernels write results straight into pinned host memory
    int list_order_horizon = 0; // COV_OPT_LIST_ORDER_HORIZON: the horizons accept stores with area_exact == 0
    std::vector<cudaEvent_t> trace_ev; // start, then per slice: h2d done, kernel start, kernel end, d2h done
    std::vector<double> trace_ms;
};

static thread_local std::string g_err_nohandle;
constexpr int kCounterSlots = 4096; // work-dispenser counters, zeroed in bulk (one fresh slot per launch)

static int fail(cov_handle *h, int code, const std::string &msg)
{
    if (h) h->err = msg;
    else g_err_nohandle = msg;
    return code;
}
static int fail_cuda(cov_handle *h, cudaError_t e, const char *what)
{
    (void)cudaGetLastError(); // clear the sticky-free error state
    return fail(h, COV_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
}
#define CK(call)                                                 \
    do {                                                         \
        cudaError_t e_ = (call);                                 \
        if (e_ != cudaSuccess) return fail_cuda(h, e_, #call);   \
    } while (0)

static int ensure(cov_handle *h, DevBuf &b, size_t bytes)
{
    if (bytes <= b.cap && b.p) return COV_OK;
    if (b.p) {
        CK(cudaStreamSynchronize(h->stream));
        CK(cudaFree(b.p));
        b.p = nullptr;
        b.cap = 0;
    }
    bytes = std::max<size_t>(bytes, 256);
    cudaError_t e = cudaMalloc(&b.p, bytes);
    if (e != cudaSuccess) {
        (void)cudaGetLastError();
        b.p = nullptr;
        return fail(h, e == cudaErrorMemoryAllocation ? COV_ERR_NOMEM : COV_ERR_CUDA,
                    std::string("cudaMalloc(") + std::to_string(bytes) + "): " + cudaGetErrorString(e));
    }
    b.cap = bytes;
    return COV_OK;
}
#define OK(call)                   \
    do {                           \
        int rc_ = (call);          \
        if (rc_ != COV_OK) return rc_; \
    } while (0)

static int ensure_pinned(cov_handle *h, void **p, size_t *cap, size_t bytes)
{
    if (*p && bytes <= *cap) return COV_OK;
    if (*p) {
        CK(cudaStreamSynchronize(h->stream));
        CK(cudaFreeHost(*p));
        *p = nullptr;
        *cap = 0;
    }
    cudaError_t e = cudaMallocHost(p, std::max<size_t>(bytes, 4096));
    if (e != cudaSuccess) {
        (void)cudaGetLastError();
        *p = nullptr;
        return fail(h, COV_ERR_NOMEM, std::string("cudaMallocHost: ") + cudaGetErrorString(e));
    }
    *cap = std::max<size_t>(bytes, 4096);
    return COV_OK;
}

static cudaEvent_t get_event(cov_handle *h)
{
    if (!h->ev_pool.empty()) {
        cudaEvent_t e = h->ev_pool.back();
        h->ev_pool.pop_back();
        return e;
    }
    cudaEvent_t e = nullptr;
    cudaEventCreate(&e);
    return e;
}
// Fold every recorded span into the running totals (synchronises the main stream).
static cudaError_t drain_spans(cov_handle *h)
{
    if (h->kernel_spans.empty()) return cudaSuccess;
    cudaError_t e = cudaStreamSynchronize(h->stream);
    if (e != cudaSuccess) return e;
    double last = 0;
    for (size_t k = 0; k < h->kernel_spans.size(); ++k) {
        float t = 0;
        e = cudaEventElapsedTime(&t, h->kernel_spans[k].first, h->kernel_spans[k].second);
        if (e != cudaSuccess) return e;
        h->drained_ms += t;
        h->drained_launches += 1;
        if (k >= h->last_call_begin) last += t;
        h->ev_pool.push_back(h->kernel_spans[k].first);
        h->ev_pool.push_back(h->kernel_spans[k].second);
    }
    h->last_call_ms_cache = last;
    h->kernel_spans.clear();
    h->last_call_begin = 0;
    return cudaSuccess;
}
// A new eval call starts: remember where its spans begin; keep the event pool bounded.
static void recycle_spans(cov_handle *h)
{
    if (h->kernel_spans.size() > 2048) (void)drain_spans(h);
    h->last_call_begin = h->kernel_spans.size();
    h->last_call_ms_cache = -1;
}

// Device-side address of pinned host memory (differs from the host address for some registered buffers);
// nullptr when the buffer cannot be written from the device.
static void *device_view(void *host)
{
    void *d = nullptr;
    if (cudaHostGetDevicePointer(&d, host, 0) != cudaSuccess) {
        (void)cudaGetLastError();
        return nullptr;
    }
    return d;
}

static bool is_pinned_host(const void *p)
{
    cudaPointerAttributes a{};
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        (void)cudaGetLastError();
        return false;
    }
    return a.type == cudaMemoryTypeHost;
}

struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int dev)
    {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        if (prev != dev) cudaSetDevice(dev);
        else prev = -1;
    }
    ~DeviceGuard()
    {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

// ------------------------------------------------------------------------------------------
// lifecycle
// ------------------------------------------------------------------------------------------
extern "C" int cov_abi_version(void) { return COV_ABI_VERSION; }

extern "C" int cov_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        (void)cudaGetLastError();
        return 0;
    }
    return n;
}

extern "C" int cov_create(int device, cov_handle **out)
{
    cov_handle *h = nullptr; // for the macros
    if (!out) return fail(nullptr, COV_ERR_INVALID, "cov_create: out is NULL");
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        (void)cudaGetLastError();
        return fail(nullptr, COV_ERR_CUDA,
                    std::string("cov_create: no usable CUDA device (") +
                        (e != cudaSuccess ? cudaGetErrorString(e) : "device count 0") +
                        "); libcoverage_cuda has no CPU fallback");
    }
    if (device < 0 || device >= n) return fail(nullptr, COV_ERR_INVALID, "cov_create: device index out of range");
    CK(cudaSetDevice(device));
    cudaDeviceProp prop{};
    CK(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10)
        return fail(nullptr, COV_ERR_CUDA,
                    std::string("cov_create: device ") + prop.name + " is sm_" + std::to_string(prop.major) +
                        std::to_string(prop.minor) + "; this library is built for sm_100a only");
    cov_handle *nh = new cov_handle();
    nh->device = device;
    h = nh;
    auto bail = [&](cudaError_t ce, const char *what) {
        int rc = fail_cuda(nullptr, ce, what);
        delete nh;
        return rc;
    };
    if ((e = cudaStreamCreateWithFlags(&nh->own_stream, cudaStreamNonBlocking)) != cudaSuccess)
        return bail(e, "cudaStreamCreate");
    if ((e = cudaStreamCreateWithFlags(&nh->s_in, cudaStreamNonBlocking)) != cudaSuccess)
        return bail(e, "cudaStreamCreate");
    if ((e = cudaStreamCreateWithFlags(&nh->s_out, cudaStreamNonBlocking)) != cudaSuccess)
        return bail(e, "cudaStreamCreate");
    nh->stream = nh->own_stream;
    nh->cfg.kernel = COV_KERNEL_AUTO;
    nh->cfg.plane_mode = -1;
    nh->cfg.num_sms = prop.multiProcessorCount;
    nh->cfg.max_smem_optin = (int)prop.sharedMemPerBlockOptin;
    if ((e = cudaMallocHost(&nh->h_small, sizeof(HostScratch))) != cudaSuccess) return bail(e, "cudaMallocHost");
    int rc = ensure(nh, nh->counter, kCounterSlots * sizeof(unsigned long long));
    if (rc == COV_OK && cudaMemset(nh->counter.p, 0, kCounterSlots * sizeof(unsigned long long)) != cudaSuccess)
        rc = fail_cuda(nh, cudaGetLastError(), "cudaMemset");
    if (rc == COV_OK) rc = ensure(nh, nh->stats, 256);
    if (rc == COV_OK) rc = ensure(nh, nh->removed, 256);
    if (rc == COV_OK) rc = ensure(nh, nh->overflow, 256);
    if (rc == COV_OK) rc = ensure(nh, nh->argmin_obj, 1024 * sizeof(double));
    if (rc == COV_OK) rc = ensure(nh, nh->argmin_idx, 1024 * sizeof(long long));
    if (rc != COV_OK) {
        g_err_nohandle = nh->err;
        delete nh;
        return rc;
    }
    *out = nh;
    return COV_OK;
}

extern "C" void cov_destroy(cov_handle *h)
{
    if (!h) return;
    DeviceGuard dg(h->device);
    cudaStreamSynchronize(h->stream);
    cudaStreamSynchronize(h->s_in);
    cudaStreamSynchronize(h->s_out);
    DevBuf *bufs[] = {&h->mult, &h->cls, &h->planes, &h->planes_q, &h->params, &h->counter, &h->stats, &h->xyT,
                      &h->small_in, &h->argmin_obj, &h->argmin_idx, &h->removed, &h->overflow, &h->dX,
                      &h->d_obj, &h->d_count, &h->d_feas, &h->d_clscnt, &h->d_prog, &h->fire[0], &h->fire[1], &h->fire_p,
                      &h->backup, &h->ent_cell, &h->ent_cls, &h->d_raw[0], &h->d_raw[1], &h->mads_in, &h->mads_out,
                      &h->ens, &h->region_discs, &h->region_arcs, &h->region_count, &h->d_area};
    for (DevBuf *b : bufs)
        if (b->p) cudaFree(b->p);
    for (int k = 0; k < 2; ++k)
        if (h->h_in[k]) cudaFreeHost(h->h_in[k]);
    if (h->h_out) cudaFreeHost(h->h_out);
    if (h->h_small) cudaFreeHost(h->h_small);
    if (h->h_poll) cudaFreeHost(h->h_poll);
    delete h->pool;
    (void)drain_spans(h);
    for (cudaEvent_t e : h->ev_pool) cudaEventDestroy(e);
    for (cudaEvent_t e : h->trace_ev) cudaEventDestroy(e);
    cudaStreamDestroy(h->s_in);
    cudaStreamDestroy(h->s_out);
    cudaStreamDestroy(h->own_stream);
    (void)cudaGetLastError();
    delete h;
}

extern "C" const char *cov_last_error(const cov_handle *h) { return h ? h->err.c_str() : g_err_nohandle.c_str(); }

extern "C" int cov_set_option(cov_handle *h, int option, int64_t value)
{
    if (!h) return fail(nullptr, COV_ERR_INVALID, "cov_set_option: NULL handle");
    switch (option) {
    case COV_OPT_KERNEL:
        if (value < COV_KERNEL_AUTO || value > COV_KERNEL_ORDERED) return fail(h, COV_ERR_INVALID, "unknown kernel id");
        h->cfg.kernel = (int)value;
        return COV_OK;
    case COV_OPT_WARPS_PER_CTA:
        if (value < 0 || value > 32) return fail(h, COV_ERR_INVALID, "warps per CTA must be 0..32");
        h->cfg.warps_per_cta = (int)value;
        return COV_OK;
    case COV_OPT_CTAS_PER_SM:
        if (value < 0 || value > 32) return fail(h, COV_ERR_INVALID, "CTAs per SM must be 0..32");
        h->cfg.ctas_per_sm = (int)value;
        return COV_OK;
    case COV_OPT_BAND_ROWS:
        if (value < 0 || value > kMaxDim) return fail(h, COV_ERR_INVALID, "band rows out of range");
        h->cfg.band_rows = (int)value;
        return COV_OK;
    case COV_OPT_FORCE_EXACT:
        h->cfg.force_exact = value != 0;
        return COV_OK;
    case COV_OPT_CHUNK:
        if (value < 0) return fail(h, COV_ERR_INVALID, "chunk must be >= 0");
        h->chunk = value;
        return COV_OK;
    case COV_OPT_TRACE:
        h->trace = value != 0;
        return COV_OK;
    case COV_OPT_ZEROCOPY_OUT:
        h->zero_copy_out = value != 0;
        return COV_OK;
    case COV_OPT_PLANE_MODE:
        if (value < -1 || value > 4) return fail(h, COV_ERR_INVALID, "plane mode must be -1..4");
        h->cfg.plane_mode = (int)value;
        return COV_OK;
    case COV_OPT_PROGRESSIVE_INDEX:
        if (value < 0 || value > kMaxUavs) return fail(h, COV_ERR_INVALID, "progressive index must be 0..1024");
        h->o.prog_which = (int)value;
        return COV_OK;
    case COV_OPT_LIST_ORDER_HORIZON:
        if (value != 0 && value != 1) return fail(h, COV_ERR_INVALID, "the list-order horizon option must be 0 or 1");
        h->list_order_horizon = (int)value;
        return COV_OK;
    }
    return fail(h, COV_ERR_INVALID, "unknown option");
}

extern "C" int cov_get_option(const cov_handle *h, int option, int64_t *value)
{
    if (!h || !value) return COV_ERR_INVALID;
    switch (option) {
    case COV_OPT_KERNEL: *value = h->cfg.kernel; return COV_OK;
    case COV_OPT_WARPS_PER_CTA: *value = h->cfg.warps_per_cta; return COV_OK;
    case COV_OPT_CTAS_PER_SM: *value = h->cfg.ctas_per_sm; return COV_OK;
    case COV_OPT_BAND_ROWS: *value = h->cfg.band_rows; return COV_OK;
    case COV_OPT_FORCE_EXACT: *value = h->cfg.force_exact; return COV_OK;
    case COV_OPT_CHUNK: *value = h->chunk; return COV_OK;
    case COV_OPT_TRACE: *value = h->trace; return COV_OK;
    case COV_OPT_ZEROCOPY_OUT: *value = h->zero_copy_out; return COV_OK;
    case COV_OPT_PLANE_MODE: *value = h->cfg.plane_mode; return COV_OK;
    case COV_OPT_PROGRESSIVE_INDEX: *value = h->o.prog_which; return COV_OK;
    case COV_OPT_LIST_ORDER_HORIZON: *value = h->list_order_horizon; return COV_OK;
    }
    return COV_ERR_INVALID;
}

extern "C" void cov_get_limits(cov_limits *out)
{
    if (!out) return;
    out->max_uavs = kMaxUavs;
    out->max_nx = kMaxDim;
    out->max_ny = kMaxDim;
    out->max_planes = kMaxPlanes;
    out->max_classes = kMaxClasses;
}

extern "C" double cov_threshold(double R) { return threshold(R); }

// ------------------------------------------------------------------------------------------
// cell store
// ------------------------------------------------------------------------------------------
static bool f32_exact(double v) { return (double)(float)v == v; }

static int check_lattice(cov_handle *h, int64_t nx, int64_t ny, double dx, double dy)
{
    if (nx < 1 || ny < 1) return fail(h, COV_ERR_INVALID, "grid: nx, ny must be >= 1");
    if (nx > kMaxDim || ny > kMaxDim) return fail(h, COV_ERR_LIMIT, "grid: nx, ny must be <= 32768");
    if (!(dx > 0) || !(dy > 0) || std::isinf(dx) || std::isinf(dy))
        return fail(h, COV_ERR_INVALID, "grid: dx, dy must be finite and > 0");
    return COV_OK;
}

static void describe_lattice(cov_handle *h, int64_t nx, int64_t ny, double dx, double dy)
{
    GridDesc &g = h->g;
    g.nx = (int)nx;
    g.ny = (int)ny;
    g.wpr = (int)((nx + 31) / 32);
    g.stride = g.wpr | 1; // odd: 32 lanes on 32 consecutive rows hit 32 different banks
    g.plane_words = (int)(((int64_t)g.ny * g.stride + 3) / 4 * 4);
    g.qstride = (g.wpr + 1) & ~1; // even, and an odd number of word pairs (see GridDesc::planes_q)
    if (((g.qstride >> 1) & 1) == 0) g.qstride += 2;
    g.planes_q = nullptr;
    g.dx = dx;
    g.dy = dy;
    g.hdx = dx / 2;
    g.hdy = dy / 2;
    g.inv_dx = 1.0 / dx;
    g.inv_dy = 1.0 / dy;
    g.dxf = (float)dx;
    g.dyf = (float)dy;
    g.hdxf = (float)g.hdx;
    g.hdyf = (float)g.hdy;
    g.inv_dxf = (float)g.inv_dx;
    g.inv_dyf = (float)g.inv_dy;
    g.extent = (float)std::max((double)nx * dx, (double)ny * dy);
    g.extent = std::nextafter(g.extent, INFINITY);
    g.k_ca = std::nextafter((float)(0.75 * g.inv_dx * 1.000001), INFINITY);
    g.lattice_f32_exact = f32_exact(dx) && f32_exact(dy) && f32_exact(g.hdx) && f32_exact(g.hdy) &&
                          f32_exact((double)nx * dx) && f32_exact((double)ny * dy);
}

// v = m * 2^e with m odd (v finite, > 0)
static void odd_decompose(double v, uint64_t &m, int &e)
{
    int ex;
    double fr = std::frexp(v, &ex); // v = fr * 2^ex, fr in [0.5, 1)
    m = (uint64_t)std::ldexp(fr, 53);
    e = ex - 53;
    while (m && !(m & 1)) {
        m >>= 1;
        ++e;
    }
}

// area_exact: every partial sum of the reference's list-order Float64 accumulation over n_entries entries of the
// classes of g is an integer multiple of a common power of two and stays below 2^53 of them, hence exact in any
// order, and so is sum_k fl(w_k * count_k).
static bool sums_exact(const GridDesc &g, int64_t n_entries)
{
    int qmin = 0;
    bool first = true;
    uint64_t ms[kMaxClasses];
    int es[kMaxClasses];
    for (int k = 0; k < g.n_classes; ++k) {
        const double w = g.class_weight[k];
        if (w == 0.0) {
            ms[k] = 0;
            es[k] = 0;
            continue;
        }
        if (!(w > 0) || std::isinf(w)) return false;
        odd_decompose(w, ms[k], es[k]);
        if (first || es[k] < qmin) qmin = es[k];
        first = false;
    }
    long double total = 0;
    for (int k = 0; k < g.n_classes; ++k)
        if (ms[k]) total += std::ldexp((long double)ms[k], es[k] - qmin) * (long double)n_entries;
    return total < 9007199254740992.0L;
}

// Derive the bit planes from the device-resident mult/cls bytes and refresh the statistics.  class_weight may be
// g.class_weight itself: each weight is read only by its own assignment below.
static int rebuild_planes(cov_handle *h, int n_classes, const double *class_weight)
{
    GridDesc &g = h->g;
    const long long ncell = (long long)g.nx * g.ny;
    unsigned long long *d_stats = (unsigned long long *)h->stats.p;
    CK(launch_grid_stats((const unsigned char *)h->mult.p, (const unsigned char *)h->cls.p, ncell, d_stats,
                         h->stream));
    h->launches += 1;
    unsigned long long *hs = h->h_small->stats;
    CK(cudaMemcpyAsync(hs, d_stats, (2 + kMaxClasses) * sizeof(unsigned long long), cudaMemcpyDeviceToHost,
                       h->stream));
    CK(cudaStreamSynchronize(h->stream));
    h->n_entries = (int64_t)hs[0];
    h->n_cells = (int64_t)hs[1];
    g.n_classes = std::max(1, n_classes);
    for (int k = 0; k < kMaxClasses; ++k) g.class_weight[k] = (k < n_classes) ? class_weight[k] : 0.0;
    int np = 0;
    for (int k = 0; k < g.n_classes; ++k) {
        const unsigned orm = (unsigned)hs[2 + k];
        for (int b = 0; b < 8; ++b)
            if (orm & (1u << b)) {
                if (np >= kMaxPlanes)
                    return fail(h, COV_ERR_LIMIT,
                                "cell store needs more than 8 bit planes (weight classes x multiplicity bits)");
                g.plane_class[np] = k;
                g.plane_mult[np] = 1 << b;
                ++np;
            }
    }
    if (np == 0) { // empty store: one all-zero plane keeps the kernels uniform
        g.plane_class[0] = 0;
        g.plane_mult[0] = 1;
        np = 1;
    }
    for (int l = np; l < kMaxPlanes; ++l) {
        g.plane_class[l] = 0;
        g.plane_mult[l] = 0;
    }
    g.n_planes = np;
    OK(ensure(h, h->planes, (size_t)np * g.plane_words * 4));
    g.planes = (const uint32_t *)h->planes.p;
    CK(launch_pack_planes((const unsigned char *)h->mult.p, (const unsigned char *)h->cls.p, g,
                          (uint32_t *)h->planes.p, h->stream));
    h->launches += 1;
    g.planes_q = nullptr;
    if (np == 1) { // the sweep mode of the CTA kernel reads plane 0 in its own aligned, swizzled layout
        OK(ensure(h, h->planes_q, ((size_t)g.ny * g.qstride + 8) * 4));
        CK(cudaMemsetAsync(h->planes_q.p, 0, ((size_t)g.ny * g.qstride + 8) * 4, h->stream));
        CK(launch_requad_plane(g, (uint32_t *)h->planes_q.p, h->stream));
        h->launches += 1;
        g.planes_q = (const uint32_t *)h->planes_q.p;
    }
    h->area_exact = sums_exact(g, h->n_entries) ? 1 : 0;
    h->have_grid = true;
    return COV_OK;
}

// ---- the ordered point list ------------------------------------------------------------------------------
static void entries_forget(cov_handle *h) // the store was re-created without a list: order = createPOI's, on demand
{
    h->ent_known = false;
    h->ent_removed_pending = false;
    h->ent_dev_valid = false;
    h->ent_cell_h.clear();
    h->ent_cls_h.clear();
    h->g.ent_cell = nullptr;
    h->g.ent_cls = nullptr;
    h->g.n_ent = 0;
}
// A setter re-creates the store (arguments checked): the automaton's state and the point list go with the old one.
static int reset_store(cov_handle *h, int64_t nx, int64_t ny, double dx, double dy)
{
    h->have_grid = false;
    h->have_fire = false;
    entries_forget(h);
    describe_lattice(h, nx, ny, dx, dy);
    OK(ensure(h, h->mult, (size_t)nx * ny + 4)); // add_points works on aligned 4-byte words
    return ensure(h, h->cls, (size_t)nx * ny + 4);
}
// Covered cells lost their entries: a known list drops them lazily (entries_apply_removals), the device list is stale.
static void entries_note_removals(cov_handle *h)
{
    h->ent_removed_pending = h->ent_known;
    h->ent_dev_valid = false;
}
// rmvCoveredPOI deletes every entry of a covered cell and keeps the order of the rest
// (src/CellFunctions.jl:81-108): drop the mirror's entries whose cell is now empty.
// m: the multiplicity bytes as they are now (host copy).
static void entries_apply_removals(cov_handle *h, const unsigned char *m)
{
    if (!h->ent_known || !h->ent_removed_pending) return;
    size_t keep = 0;
    for (size_t p = 0; p < h->ent_cell_h.size(); ++p)
        if (m[(size_t)h->ent_cell_h[p]]) {
            h->ent_cell_h[keep] = h->ent_cell_h[p];
            h->ent_cls_h[keep] = h->ent_cls_h[p];
            ++keep;
        }
    h->ent_cell_h.resize(keep);
    h->ent_cls_h.resize(keep);
    h->ent_removed_pending = false;
    h->ent_dev_valid = false;
}
static int entries_apply_removals(cov_handle *h)
{
    if (!h->ent_known || !h->ent_removed_pending) return COV_OK;
    const size_t ncell = (size_t)h->g.nx * h->g.ny;
    std::vector<unsigned char> m(ncell);
    CK(cudaMemcpyAsync(m.data(), h->mult.p, ncell, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    entries_apply_removals(h, m.data());
    return COV_OK;
}
// The host list of a store that no list was ever given for (bit grid, cell bytes, createPOI, automaton), built from
// the cell store as it is now: createPOI's order, i outer and j inner (src/AreaCoverageCalculation.jl:14-15), the
// entries of a cell together.
static void entries_from_cells(cov_handle *h, const unsigned char *m, const unsigned char *k)
{
    h->ent_cell_h.clear();
    h->ent_cls_h.clear();
    for (int i = 0; i < h->g.nx; ++i)
        for (int j = 0; j < h->g.ny; ++j) {
            const size_t cell = (size_t)i + (size_t)h->g.nx * j;
            for (unsigned r = 0; r < m[cell]; ++r) {
                h->ent_cell_h.push_back((int)cell);
                h->ent_cls_h.push_back((unsigned char)(k[cell] & (kMaxClasses - 1)));
            }
        }
}
static int entries_from_cells(cov_handle *h)
{
    const size_t ncell = (size_t)h->g.nx * h->g.ny;
    std::vector<unsigned char> m(ncell), k(ncell);
    CK(cudaMemcpyAsync(m.data(), h->mult.p, ncell, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(k.data(), h->cls.p, ncell, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    entries_from_cells(h, m.data(), k.data());
    return COV_OK;
}
// Make g.ent_cell / g.ent_cls / g.n_ent describe the current list on the device.
static int entries_on_device(cov_handle *h)
{
    if (h->ent_dev_valid) return COV_OK;
    OK(entries_apply_removals(h));
    if (!h->ent_known) OK(entries_from_cells(h));
    const size_t P = h->ent_cell_h.size();
    if ((int64_t)P != h->n_entries)
        return fail(h, COV_ERR_STATE, "internal: the ordered point list disagrees with the cell store (" +
                                          std::to_string(P) + " vs " + std::to_string(h->n_entries) + " entries)");
    OK(ensure(h, h->ent_cell, std::max<size_t>(P, 1) * sizeof(int)));
    OK(ensure(h, h->ent_cls, std::max<size_t>(P, 1)));
    if (P) {
        CK(cudaMemcpyAsync(h->ent_cell.p, h->ent_cell_h.data(), P * sizeof(int), cudaMemcpyHostToDevice, h->stream));
        CK(cudaMemcpyAsync(h->ent_cls.p, h->ent_cls_h.data(), P, cudaMemcpyHostToDevice, h->stream));
        CK(cudaStreamSynchronize(h->stream)); // pageable sources
    }
    if (!h->ent_known) { // the canonical list is cheap to rebuild and can be large: do not keep it
        h->ent_cell_h.clear();
        h->ent_cell_h.shrink_to_fit();
        h->ent_cls_h.clear();
        h->ent_cls_h.shrink_to_fit();
    }
    h->g.ent_cell = (const int *)h->ent_cell.p;
    h->g.ent_cls = (const unsigned char *)h->ent_cls.p;
    h->g.n_ent = (long long)P;
    h->ent_dev_valid = true;
    return COV_OK;
}

// An append (cov_add_points, cov_fire_step) can fail half-way: a multiplicity overflowing 255 or entries of
// different weights on one cell are found by the kernel that is already writing.  The store is snapshot
// before and put back on failure, so that mult/cls, the bit planes and n_entries never disagree.
static int snapshot_cells(cov_handle *h)
{
    const size_t ncell = (size_t)h->g.nx * h->g.ny + 4;
    OK(ensure(h, h->backup, 2 * ncell));
    CK(cudaMemcpyAsync(h->backup.p, h->mult.p, ncell, cudaMemcpyDeviceToDevice, h->stream));
    CK(cudaMemcpyAsync((char *)h->backup.p + ncell, h->cls.p, ncell, cudaMemcpyDeviceToDevice, h->stream));
    return COV_OK;
}
static void restore_cells(cov_handle *h)
{
    const size_t ncell = (size_t)h->g.nx * h->g.ny + 4;
    cudaError_t e = cudaMemcpyAsync(h->mult.p, h->backup.p, ncell, cudaMemcpyDeviceToDevice, h->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(h->cls.p, (char *)h->backup.p + ncell, ncell, cudaMemcpyDeviceToDevice, h->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
    if (e != cudaSuccess) { // cannot vouch for the store any more: make the next evaluation fail loudly
        (void)cudaGetLastError();
        h->have_grid = false;
    }
}

extern "C" int cov_set_grid_bits(cov_handle *h, int64_t nx, int64_t ny, double dx, double dy,
                                 const uint32_t *bits, double weight)
{
    if (!h) return fail(nullptr, COV_ERR_INVALID, "NULL handle");
    DeviceGuard dg(h->device);
    if (!bits) return fail(h, COV_ERR_INVALID, "cov_set_grid_bits: bits is NULL");
    OK(check_lattice(h, nx, ny, dx, dy));
    OK(reset_store(h, nx, ny, dx, dy));
    const size_t words = (size_t)ny * ((nx + 31) / 32);
    DevBuf tmp;
    OK(ensure(h, tmp, words * 4));
    cudaError_t e = cudaMemcpyAsync(tmp.p, bits, words * 4, cudaMemcpyHostToDevice, h->stream);
    if (e == cudaSuccess)
        e = launch_bits_to_cells((const uint32_t *)tmp.p, (int)nx, (int)ny, (unsigned char *)h->mult.p,
                                 (unsigned char *)h->cls.p, h->stream);
    h->launches += 1;
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
    cudaFree(tmp.p);
    if (e != cudaSuccess) return fail_cuda(h, e, "cov_set_grid_bits");
    return rebuild_planes(h, 1, &weight);
}

extern "C" int cov_set_grid_cells(cov_handle *h, int64_t nx, int64_t ny, double dx, double dy,
                                  const uint8_t *mult, const uint8_t *cls, int64_t n_classes,
                                  const double *class_weight)
{
    if (!h) return fail(nullptr, COV_ERR_INVALID, "NULL handle");
    DeviceGuard dg(h->device);
    if (!mult || !class_weight) return fail(h, COV_ERR_INVALID, "cov_set_grid_cells: NULL argument");
    if (n_classes < 1 || n_classes > kMaxClasses)
        return fail(h, COV_ERR_LIMIT, "cov_set_grid_cells: n_classes must be 1..4");
    OK(check_lattice(h, nx, ny, dx, dy));
    const size_t ncell = (size_t)nx * ny;
    if (cls)
        for (size_t t = 0; t < ncell; ++t)
            if (cls[t] >= n_classes) return fail(h, COV_ERR_INVALID, "cov_set_grid_cells: class index out of range");
    OK(reset_store(h, nx, ny, dx, dy));
    CK(cudaMemcpyAsync(h->mult.p, mult, ncell, cudaMemcpyHostToDevice, h->stream));
    if (cls) CK(cudaMemcpyAsync(h->cls.p, cls, ncell, cudaMemcpyHostToDevice, h->stream));
    else CK(cudaMemsetAsync(h->cls.p, 0, ncell, h->stream));
    CK(launch_normalize_cls((const unsigned char *)h->mult.p, (unsigned char *)h->cls.p, (long long)ncell, h->stream));
    h->launches += 1;
    CK(cudaStreamSynchronize(h->stream));
    return rebuild_planes(h, (int)n_classes, class_weight);
}

extern "C" int cov_set_grid_full(cov_handle *h, int64_t nx, int64_t ny, double dx, double dy)
{
    if (!h) return fail(nullptr, COV_ERR_INVALID, "NULL handle");
    DeviceGuard dg(h->device);
    OK(check_lattice(h, nx, ny, dx, dy));
    OK(reset_store(h, nx, ny, dx, dy));
    CK(launch_fill_full((unsigned char *)h->mult.p, (unsigned char *)h->cls.p, (long long)nx * ny, h->stream));
    h->launches += 1;
    const double w = dx * dy; // createPOI: area = weight = dx*dy
    return rebuild_planes(h, 1, &w);
}

// Map list entries onto the lattice (bit-exact centre check) and weight classes.
static int map_points(cov_handle *h, const double *pts5, int64_t P, std::vector<int> &cell,
                      std::vector<unsigned char> &pcls, int &n_classes, double *class_weight)
{
    const GridDesc &g = h->g;
    cell.resize((size_t)P);
    pcls.resize((size_t)P);
    for (int64_t p = 0; p < P; ++p) {
        const double x = pts5[5 * p], y = pts5[5 * p + 1], w = pts5[5 * p + 3];
        const double fi = std::nearbyint((x + g.hdx) / g.dx), fj = std::nearbyint((y + g.hdy) / g.dy);
        bool ok = fi >= 1 && fi <= g.nx && fj >= 1 && fj <= g.ny;
        if (ok) {
            volatile double cx = fi * g.dx; // individually rounded, as the reference forms them
            volatile double cy = fj * g.dy;
            ok = (cx - g.hdx == x) && (cy - g.hdy == y);
        }
        if (!ok) {
            char buf[160];
            snprintf(buf, sizeof buf, "point %lld (%.17g, %.17g) is not a cell centre of the %dx%d lattice",
                     (long long)p, x, y, g.nx, g.ny);
            return fail(h, COV_ERR_OFF_LATTICE, buf);
        }
        int k = -1;
        for (int q = 0; q < n_classes; ++q)
            if (class_weight[q] == w) {
                k = q;
                break;
            }
        if (k < 0) {
            if (w != w) return fail(h, COV_ERR_INVALID, "point weight is NaN");
            if (n_classes >= kMaxClasses)
                return fail(h, COV_ERR_LIMIT, "more than 4 distinct point weights");
            k = n_classes;
            class_weight[n_classes++] = w;
        }
        cell[(size_t)p] = ((int)fi - 1) + g.nx * ((int)fj - 1);
        pcls[(size_t)p] = (unsigned char)k;
    }
    return COV_OK;
}

static int upload_points(cov_handle *h, const std::vector<int> &cell, const std::vector<unsigned char> &pcls)
{
    const size_t P = cell.size();
    if (P == 0) return COV_OK;
    DevBuf dcell, dcls;
    int rc = ensure(h, dcell, P * sizeof(int));
    if (rc == COV_OK) rc = ensure(h, dcls, P);
    cudaError_t e = cudaSuccess;
    int *hov = &h->h_small->overflow;
    if (rc == COV_OK) {
        e = cudaMemcpyAsync(dcell.p, cell.data(), P * sizeof(int), cudaMemcpyHostToDevice, h->stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(dcls.p, pcls.data(), P, cudaMemcpyHostToDevice, h->stream);
        if (e == cudaSuccess) e = cudaMemsetAsync(h->overflow.p, 0, sizeof(int), h->stream);
        if (e == cudaSuccess)
            e = launch_add_points((unsigned char *)h->mult.p, (unsigned char *)h->cls.p, (const int *)dcell.p,
                                  (const unsigned char *)dcls.p, (long long)P, (int *)h->overflow.p, h->stream);
        h->launches += 1;
        if (e == cudaSuccess)
            e = cudaMemcpyAsync(hov, h->overflow.p, sizeof(int), cudaMemcpyDeviceToHost, h->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
    }
    if (dcell.p) cudaFree(dcell.p);
    if (dcls.p) cudaFree(dcls.p);
    if (rc != COV_OK) return rc;
    if (e != cudaSuccess) return fail_cuda(h, e, "upload_points");
    if (*hov == 1) return fail(h, COV_ERR_LIMIT, "more than 255 list entries on one cell");
    if (*hov == 2) return fail(h, COV_ERR_INVALID, "entries on one cell carry different weights");
    return COV_OK;
}

extern "C" int cov_set_points(cov_handle *h, const double *pts5, int64_t P, int64_t nx, int64_t ny, double dx,
                              double dy)
{
    if (!h) return fail(nullptr, COV_ERR_INVALID, "NULL handle");
    DeviceGuard dg(h->device);
    if (P < 0 || (P > 0 && !pts5)) return fail(h, COV_ERR_INVALID, "cov_set_points: bad list");
    OK(check_lattice(h, nx, ny, dx, dy));
    OK(reset_store(h, nx, ny, dx, dy));
    std::vector<int> cell;
    std::vector<unsigned char> pcls;
    int n_classes = 0;
    double cw[kMaxClasses] = {0, 0, 0, 0};
    OK(map_points(h, pts5, P, cell, pcls, n_classes, cw));
    if (n_classes == 0) {
        n_classes = 1;
        cw[0] = dx * dy;
    }
    const size_t ncell = (size_t)nx * ny;
    CK(cudaMemsetAsync(h->mult.p, 0, ncell + 4, h->stream));
    CK(cudaMemsetAsync(h->cls.p, 0xff, ncell + 4, h->stream));
    OK(upload_points(h, cell, pcls));
    h->ent_cell_h = cell; // the list order of the reference's points_of_interest
    h->ent_cls_h = pcls;
    h->ent_known = true;
    return rebuild_planes(h, n_classes, cw);
}

extern "C" int cov_add_points(cov_handle *h, const double *pts5, int64_t P)
{
    if (!h) return fail(nullptr, COV_ERR_INVALID, "NULL handle");
    DeviceGuard dg(h->device);
    if (!h->have_grid) return fail(h, COV_ERR_STATE, "cov_add_points: no grid set");
    if (P < 0 || (P > 0 && !pts5)) return fail(h, COV_ERR_INVALID, "cov_add_points: bad list");
    std::vector<int> cell;
    std::vector<unsigned char> pcls;
    int n_classes = h->g.n_classes;
    double cw[kMaxClasses];
    for (int k = 0; k < kMaxClasses; ++k) cw[k] = h->g.class_weight[k];
    if (h->n_entries == 0) n_classes = 0; // an empty store has no weight yet
    OK(map_points(h, pts5, P, cell, pcls, n_classes, cw));
    if (n_classes == 0) {
        n_classes = 1;
        cw[0] = h->g.class_weight[0];
    }
    OK(entries_apply_removals(h)); // before new entries can land on cells that a removal emptied
    if (!h->ent_known) {
        // push! appends after every entry already in the list, whatever setter built it: fix the order of the
        // store as it is (createPOI's) before the new entries land on its cells, and keep the list from here on
        OK(entries_from_cells(h));
        h->ent_known = true;
    }
    OK(snapshot_cells(h));
    const int rc = upload_points(h, cell, pcls);
    if (rc != COV_OK) { // nothing was appended: the store, its planes and its counts stay as they were
        const std::string msg = h->err;
        restore_cells(h);
        h->err = msg;
        return rc;
    }
    // push! appends at the end (src/CellFunctions.jl:74)
    const size_t old_len = h->ent_cell_h.size();
    const int old_classes = h->g.n_classes;
    double old_cw[kMaxClasses];
    for (int k = 0; k < kMaxClasses; ++k) old_cw[k] = h->g.class_weight[k];
    h->ent_cell_h.insert(h->ent_cell_h.end(), cell.begin(), cell.end());
    h->ent_cls_h.insert(h->ent_cls_h.end(), pcls.begin(), pcls.end());
    h->ent_dev_valid = false;
    const int rc_planes = rebuild_planes(h, n_classes, cw);
    if (rc_planes != COV_OK) { // more bit planes than the kernels sweep: put the store back as it was
        const std::string msg = h->err;
        restore_cells(h);
        h->ent_cell_h.resize(old_len);
        h->ent_cls_h.resize(old_len);
        if (h->have_grid && rebuild_planes(h, old_classes, old_cw) != COV_OK) h->have_grid = false;
        h->err = msg;
        return rc_planes;
    }
    return COV_OK;
}

extern "C" int cov_get_grid_info(const cov_handle *h, cov_grid_info *info)
{
    if (!h || !info) return COV_ERR_INVALID;
    if (!h->have_grid) return COV_ERR_STATE;
    info->nx = h->g.nx;
    info->ny = h->g.ny;
    info->dx = h->g.dx;
    info->dy = h->g.dy;
    info->n_entries = h->n_entries;
    info->n_cells = h->n_cells;
    info->n_planes = h->g.n_planes;
    info->n_classes = h->g.n_classes;
    info->area_exact = h->area_exact;
    info->planes_in_smem = span_small_applies(h->g, h->have_params ? h->o.N : 1, h->cfg, 0, nullptr, nullptr) ? 1 : 0;
    return COV_OK;
}

extern "C" int cov_get_class_weights(const cov_handle *h, double *class_weight, int64_t cap)
{
    if (!h || !class_weight) return COV_ERR_INVALID;
    if (!h->have_grid) return COV_ERR_STATE;
    for (int64_t k = 0; k < cap && k < h->g.n_classes; ++k) class_weight[k] = h->g.class_weight[k];
    return COV_OK;
}

extern "C" int cov_get_grid_cells(cov_handle *h, uint8_t *mult)
{
    if (!h) return fail(nullptr, COV_ERR_INVALID, "NULL handle");
    DeviceGuard dg(h->device);
    if (!h->have_grid) return fail(h, COV_ERR_STATE, "no grid set");
    if (!mult) return fail(h, COV_ERR_INVALID, "NULL output");
    CK(cudaMemcpyAsync(mult, h->mult.p, (size_t)h->g.nx * h->g.ny, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return COV_OK;
}

// discs [x;y;R] -> device [x;y;T(R)]
static int upload_discs_T(cov_handle *h, const double *xyR, int64_t N)
{
    if (N < 1 || N > kMaxUavs) return fail(h, COV_ERR_LIMIT, "N must be 1..1024");
    if (!xyR) return fail(h, COV_ERR_INVALID, "NULL disc vector");
    OK(ensure(h, h->xyT, (size_t)3 * N * 8));
    OK(ensure(h, h->small_in, (size_t)3 * N * 8));
    CK(cudaMemcpyAsync(h->small_in.p, xyR, (size_t)3 * N * 8, cudaMemcpyHostToDevice, h->stream));
    CK(launch_thresholds((const double *)h->small_in.p, (int)N, (double *)h->xyT.p, h->stream));
    h->launches += 1;
    return COV_OK;
}

extern "C" int cov_remove_covered(cov_handle *h, const double *xyR, int64_t N, int64_t *removed)
{
    if (!h) return fail(nullptr, COV_ERR_INVALID, "NULL handle");
    DeviceGuard dg(h->device);
    if (!h->have_grid) return fail(h, COV_ERR_STATE, "cov_remove_covered: no grid set");
    OK(upload_discs_T(h, xyR, N));
    CK(launch_remove_covered((unsigned char *)h->mult.p, (unsigned char *)h->cls.p, h->g, (const double *)h->xyT.p, (int)N,
                             (unsigned long long *)h->removed.p, h->stream));
    h->launches += 1;
    unsigned long long *hr = &h->h_small->removed;
    CK(cudaMemcpyAsync(hr, h->removed.p, sizeof(unsigned long long), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if (removed) *removed = (int64_t)*hr;
    if (*hr) entries_note_removals(h);
    return rebuild_planes(h, h->g.n_classes, h->g.class_weight);
}

extern "C" int cov_covered_mask(cov_handle *h, const double *x, uint8_t *mask)
{
    if (!h) return fail(nullptr, COV_ERR_INVALID, "NULL handle");
    DeviceGuard dg(h->device);
    if (!h->have_grid || !h->have_params) return fail(h, COV_ERR_STATE, "cov_covered_mask: grid/params not set");
    if (!mask) return fail(h, COV_ERR_INVALID, "NULL output");
    OK(upload_discs_T(h, x, h->o.N));
    const size_t ncell = (size_t)h->g.nx * h->g.ny;
    DevBuf dm;
    OK(ensure(h, dm, ncell));
    cudaError_t e = launch_covered_mask((unsigned char *)dm.p, h->g, (const double *)h->xyT.p, h->o.N, h->stream);
    h->launches += 1;
    if (e == cudaSuccess) e = cudaMemcpyAsync(mask, dm.p, ncell, cudaMemcpyDeviceToHost, h->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
    cudaFree(dm.p);
    if (e != cudaSuccess) return fail_cuda(h, e, "cov_covered_mask");
    return COV_OK;
}


// ------------------------------------------------------------------------------------------
// forest-fire automaton (src/DynamicArea.jl of the reference) feeding the cell store directly
// ------------------------------------------------------------------------------------------
extern "C" int cov_fire_init(cov_handle *h, int64_t nx, int64_t ny, double dx, double dy, const uint8_t *state,
                             int32_t push_initial)
{
    if (!h) return fail(nullptr, COV_ERR_INVALID, "NULL handle");
    DeviceGuard dg(h->device);
    if (!state) return fail(h, COV_ERR_INVALID, "cov_fire_init: state is NULL");
    OK(check_lattice(h, nx, ny, dx, dy));
    const size_t ncell = (size_t)nx * ny;
    for (size_t t = 0; t < ncell; ++t)
        if (state[t] > 2) return fail(h, COV_ERR_INVALID, "cov_fire_init: cell states must be 0 (empty), 1 (tree), 2 (fire)");
    OK(reset_store(h, nx, ny, dx, dy));
    OK(ensure(h, h->fire[0], ncell));
    OK(ensure(h, h->fire[1], ncell));
    OK(ensure(h, h->fire_p, 9 * sizeof(double)));
    CK(cudaMemcpyAsync(h->fire[0].p, state, ncell, cudaMemcpyHostToDevice, h->stream));
    CK(launch_fire_seed((const unsigned char *)h->fire[0].p, (unsigned char *)h->mult.p, (unsigned char *)h->cls.p,
                        (long long)ncell, push_initial, h->stream));
    h->launches += 1;
    CK(cudaStreamSynchronize(h->stream));
    h->fire_cur = 0;
    h->have_fire = true;
    const double w = dx * dy; // DynamicArea.jl:65: area = weight = dx*dy
    return rebuild_planes(h, 1, &w);
}

// The probability of ignition from the neighbour at window index (a, b), a, b = 1..3, exactly as the reference forms
// it: wind_speed * cos(wind_direction - atan(2-b, 2-a)) * prob_spread, to hp[(a-1) + 3(b-1)].
static void fire_probs(double wind_speed, double wind_direction, double prob_spread, double *hp)
{
    for (int b = 1; b <= 3; ++b)
        for (int a = 1; a <= 3; ++a) {
            volatile double ang = atan2((double)(2 - b), (double)(2 - a));
            volatile double c = cos(wind_direction - ang);
            volatile double p = wind_speed * c;
            hp[(a - 1) + 3 * (b - 1)] = p * prob_spread;
        }
}

// cov_fire_step's preconditions on the store (cov_run_horizon_fire shares them).
static int check_fire_store(cov_handle *h, const char *who)
{
    if (!h->have_fire) return fail(h, COV_ERR_STATE, std::string(who) + ": cov_fire_init has not been called");
    if (h->g.n_classes != 1)
        return fail(h, COV_ERR_STATE, std::string(who) + ": the cell store holds several weight classes");
    if (h->g.class_weight[0] != h->g.dx * h->g.dy) // DynamicArea.jl:65: every pushed entry weighs dx*dy
        return fail(h, COV_ERR_STATE, std::string(who) + ": the cell store's weight class is not dx*dy, the weight "
                                                          "the automaton pushes");
    return COV_OK;
}

extern "C" int cov_fire_step(cov_handle *h, double wind_speed, double wind_direction, double prob_spread,
                             uint64_t seed, int64_t step, int32_t append, int64_t *n_pushed)
{
    if (!h) return fail(nullptr, COV_ERR_INVALID, "NULL handle");
    DeviceGuard dg(h->device);
    if (!h->have_fire) return fail(h, COV_ERR_STATE, "cov_fire_step: cov_fire_init has not been called");
    if (step < 0 || step > 0xffffffffll) return fail(h, COV_ERR_INVALID, "cov_fire_step: step out of range");
    OK(check_fire_store(h, "cov_fire_step"));
    double *hp = h->h_small->fire_p;
    fire_probs(wind_speed, wind_direction, prob_spread, hp);
    CK(cudaMemcpyAsync(h->fire_p.p, hp, 9 * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemsetAsync(h->removed.p, 0, sizeof(unsigned long long), h->stream));
    CK(cudaMemsetAsync(h->overflow.p, 0, sizeof(int), h->stream));
    if (append) OK(snapshot_cells(h));
    const int cur = h->fire_cur;
    CK(launch_fire_step((const unsigned char *)h->fire[cur].p, (unsigned char *)h->fire[cur ^ 1].p,
                        (unsigned char *)h->mult.p, (unsigned char *)h->cls.p, h->g.nx, h->g.ny, seed,
                        (unsigned int)step, (const double *)h->fire_p.p, append, (unsigned long long *)h->removed.p,
                        (int *)h->overflow.p, h->stream));
    h->launches += 1;
    unsigned long long *hr = &h->h_small->removed;
    int *hov = &h->h_small->overflow;
    CK(cudaMemcpyAsync(hr, h->removed.p, sizeof(unsigned long long), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(hov, h->overflow.p, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if (*hov) { // the step did not happen: automaton state and cell store stay as they were
        if (append) restore_cells(h);
        if (n_pushed) *n_pushed = 0;
        return fail(h, COV_ERR_LIMIT, "more than 255 list entries on one cell");
    }
    h->fire_cur = cur ^ 1;
    if (n_pushed) *n_pushed = (int64_t)*hr;
    if (!append || *hr == 0) return COV_OK;
    // The automaton pushes in cell order; from here on the list order is createPOI's.  The store has one weight
    // class, so every covered entry adds the same weight and the list-order sum is the same in any order.
    entries_forget(h);
    return rebuild_planes(h, 1, h->g.class_weight);
}

extern "C" int cov_fire_get_state(cov_handle *h, uint8_t *state)
{
    if (!h) return fail(nullptr, COV_ERR_INVALID, "NULL handle");
    DeviceGuard dg(h->device);
    if (!h->have_fire) return fail(h, COV_ERR_STATE, "cov_fire_get_state: cov_fire_init has not been called");
    if (!state) return fail(h, COV_ERR_INVALID, "NULL output");
    CK(cudaMemcpyAsync(state, h->fire[h->fire_cur].p, (size_t)h->g.nx * h->g.ny, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return COV_OK;
}

// ------------------------------------------------------------------------------------------
// parameters
// ------------------------------------------------------------------------------------------
extern "C" int cov_set_params(cov_handle *h, int64_t N, const double *r_max, double penalty_scale,
                              const double *prev_xyR, const double *d_lim, double tan_half_fov, double sep_min,
                              int32_t use_cons7)
{
    if (!h) return fail(nullptr, COV_ERR_INVALID, "NULL handle");
    DeviceGuard dg(h->device);
    if (N < 1 || N > kMaxUavs) return fail(h, COV_ERR_LIMIT, "cov_set_params: N must be 1..1024");
    if (!r_max) return fail(h, COV_ERR_INVALID, "cov_set_params: r_max is NULL");
    if (prev_xyR && !d_lim) return fail(h, COV_ERR_INVALID, "cov_set_params: d_lim is NULL while prev_xyR is set");
    std::vector<double> hp((size_t)5 * N, 0.0);
    for (int64_t i = 0; i < N; ++i) hp[i] = r_max[i];
    if (prev_xyR)
        for (int64_t i = 0; i < N; ++i) {
            hp[N + i] = prev_xyR[i];
            hp[2 * N + i] = prev_xyR[N + i];
            volatile double z = prev_xyR[2 * N + i] / tan_half_fov; // z1 = pre.R / tan(FOV/2)
            hp[3 * N + i] = z;
            hp[4 * N + i] = threshold_ge(d_lim[i]);
        }
    OK(ensure(h, h->params, (size_t)5 * N * 8));
    // pageable source: the copy is staged before the call returns, hp may go out of scope
    CK(cudaMemcpyAsync(h->params.p, hp.data(), (size_t)5 * N * 8, cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    ObjParams &o = h->o;
    o.N = (int)N;
    o.use_cons3 = prev_xyR != nullptr;
    o.use_cons7 = use_cons7 != 0;
    o.use_cons8 = sep_min > 0;
    o.penalty_scale = penalty_scale;
    o.tan_half_fov = tan_half_fov;
    {
        volatile double c7 = 19 * tan_half_fov;
        o.cons7_R = c7;
    }
    o.sep_T = o.use_cons8 ? threshold(sep_min) : 0.0;
    const double *base = (const double *)h->params.p;
    o.r_max = base;
    o.prev_x = base + N;
    o.prev_y = base + 2 * N;
    o.prev_z = base + 3 * N;
    o.cons3_G = base + 4 * N;
    h->have_params = true;
    return COV_OK;
}

// ------------------------------------------------------------------------------------------
// evaluation
// ------------------------------------------------------------------------------------------
// A fresh zeroed slot of the counter ring (the work dispenser of one launch on the main stream).
static int take_counter(cov_handle *h, unsigned long long **counter)
{
    if (h->counter_next >= kCounterSlots) { // ring used up: zero it again (stream-ordered after its last user)
        CK(cudaMemsetAsync(h->counter.p, 0, kCounterSlots * sizeof(unsigned long long), h->stream));
        h->counter_next = 0;
    }
    *counter = (unsigned long long *)h->counter.p + h->counter_next++;
    return COV_OK;
}

// One kernel launch on the main stream; timed: inside a (start, stop) event pair for cov_last_kernel_ms, with the
// counter slot (when asked for) taken inside it.  cudaErrorInvalidConfiguration is COV_ERR_LIMIT with limit_msg.
template <class Launch>
static int timed_launch(cov_handle *h, bool timed, unsigned long long **counter, const char *what, const char *limit_msg,
                        Launch &&launch)
{
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    if (timed) {
        e0 = get_event(h);
        e1 = get_event(h);
        CK(cudaEventRecord(e0, h->stream));
    }
    const int rc = counter ? take_counter(h, counter) : COV_OK;
    const cudaError_t e = rc == COV_OK ? launch() : cudaSuccess;
    if (rc != COV_OK || e != cudaSuccess) {
        if (timed) {
            h->ev_pool.push_back(e0);
            h->ev_pool.push_back(e1);
        }
        if (rc != COV_OK) return rc;
        if (e != cudaErrorInvalidConfiguration) return fail_cuda(h, e, what);
        (void)cudaGetLastError();
        return fail(h, COV_ERR_LIMIT, limit_msg);
    }
    h->launches += 1;
    if (timed) {
        CK(cudaEventRecord(e1, h->stream));
        h->kernel_spans.emplace_back(e0, e1);
    }
    return COV_OK;
}

static int launch_on_main(cov_handle *h, const double *dX, int64_t B, const EvalOut &out, bool timed)
{
    h->cfg.ordered = h->area_exact ? 0 : 1; // non-dyadic weights: the sum is replayed in list order
    if (h->cfg.ordered || h->cfg.kernel == COV_KERNEL_ORDERED) OK(entries_on_device(h));
    unsigned long long *counter = nullptr;
    return timed_launch(h, timed, &counter, "coverage kernel launch",
                        "grid row / N too large for the shared-memory plan of this kernel", [&] {
                            return launch_eval(h->g, h->o, h->cfg, dX, (long long)B, out, counter, h->stream, &h->last_info);
                        });
}

static int check_ready(cov_handle *h, const char *who)
{
    if (!h->have_grid) return fail(h, COV_ERR_STATE, std::string(who) + ": no grid set");
    if (!h->have_params) return fail(h, COV_ERR_STATE, std::string(who) + ": no parameters set");
    return COV_OK;
}

// Candidates per device window: as many as fit cap_bytes, at least one.
static int64_t window_rows(int64_t B, size_t row_bytes, size_t cap_bytes)
{
    return std::max<int64_t>(1, std::min<int64_t>(std::max<int64_t>(B, 1), (int64_t)(cap_bytes / row_bytes)));
}

// The poll winner: the lowest objective, a tie to the earlier index; no winner is (INFINITY, -1).  offer: candidate i
// (< 0: none) of a window or shard that starts at candidate base.
struct Winner {
    double obj = INFINITY;
    int64_t idx = -1;
    void offer(double o, int64_t i, int64_t base = 0)
    {
        if (i >= 0 && (idx < 0 || o < obj)) {
            obj = o;
            idx = base + i;
        }
    }
};
// Enqueue the winner of one device window (objectives, feasibility flags, wn candidates) and its 16 bytes' way home;
// once the main stream is synchronised, offer h_small->win_obj / win_idx.
static int enqueue_winner(cov_handle *h, const double *d_obj, const unsigned char *d_feas, int64_t wn, int barrier)
{
    CK(launch_argmin(d_obj, d_feas, wn, barrier, (double *)h->argmin_obj.p, (long long *)h->argmin_idx.p, 1024,
                     h->stream));
    h->launches += 2;
    CK(cudaMemcpyAsync(&h->h_small->win_obj, h->argmin_obj.p, 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(&h->h_small->win_idx, h->argmin_idx.p, 8, cudaMemcpyDeviceToHost, h->stream));
    return COV_OK;
}

extern "C" int cov_eval_batch_device(cov_handle *h, const double *dX, int64_t B, double *d_obj, int64_t *d_count,
                                     uint8_t *d_feasible)
{
    if (!h) return fail(nullptr, COV_ERR_INVALID, "NULL handle");
    DeviceGuard dg(h->device);
    OK(check_ready(h, "cov_eval_batch_device"));
    if (B < 0 || (B > 0 && (!dX || !d_obj))) return fail(h, COV_ERR_INVALID, "cov_eval_batch_device: bad arguments");
    if (B == 0) return COV_OK;
    recycle_spans(h);
    EvalOut out{};
    out.obj = d_obj;
    out.count = (long long *)d_count;
    out.feasible = d_feasible;
    return launch_on_main(h, dX, B, out, true);
}

// The host pipeline: candidates are cut into slices; slice k's H2D copy (stream s_in), the kernel
// of slice k-1 (main stream) and the D2H copy of slice k-2's results (stream s_out) overlap.
// Pageable host buffers go through two pinned staging buffers; pinned ones are DMA'd in place.
static void host_copy(cov_handle *h, void *dst, const void *src, size_t bytes)
{
    static const size_t pool_min = [] {
        const char *e = getenv("COV_POOL_MIN_BYTES"); // experiments; default: from 1 MiB on
        return e ? (size_t)strtoull(e, nullptr, 10) : (size_t)(1u << 20);
    }();
    if (bytes >= pool_min) {
        if (!h->pool) {
            const unsigned hc = std::thread::hardware_concurrency();
            const char *e = getenv("COV_POOL_THREADS"); // experiments; default: up to 7 workers + the calling thread
            const unsigned want = e ? (unsigned)atoi(e) : 7u;
            h->pool = new CopyPool((int)std::min(std::max(want, 1u), std::max(2u, hc) - 1u));
        }
        h->pool->copy(dst, src, bytes);
    } else {
        memcpy(dst, src, bytes);
    }
}

// The per-candidate results of a host-path call, in the order of every packed layout: the 8-byte columns before the
// 1-byte feasibility flags, which keeps each column of a packed block 8-byte aligned.
enum { COL_OBJ, COL_COUNT, COL_CLS, COL_PROG, COL_FEAS, kCols };
struct Col {
    char *host;           // the caller's buffer; null: not requested
    size_t row;           // bytes per candidate
    DevBuf *dev;          // the column of the device window
    bool pinned = false;  // host is null or pinned: written in place, not staged
    size_t at = 0;        // offset in a packed layout (the small path's scratch, the staging block)
};
using Cols = Col[kCols];

// Lays the requested columns that are not pinned one after the other, n candidates each; returns the bytes.
static size_t pack_cols(Cols &c, size_t n)
{
    size_t bytes = 0;
    for (Col &col : c)
        if (col.host && !col.pinned) {
            col.at = bytes;
            bytes += n * col.row;
        }
    return bytes;
}
static EvalOut eval_out(char *const at[kCols])
{
    EvalOut out{};
    out.obj = (double *)at[COL_OBJ];
    out.count = (long long *)at[COL_COUNT];
    out.class_count = (long long *)at[COL_CLS];
    out.progressive = (double *)at[COL_PROG];
    out.feasible = (unsigned char *)at[COL_FEAS];
    return out;
}
// Device views of the host homes (pinned buffer, or staging block so) of the requested columns of the slice from
// candidate g0 (c0 in its window); false when the device cannot address one.
static bool view_cols(const Cols &c, char *so, int64_t g0, int64_t c0, char *at[kCols])
{
    for (int k = 0; k < kCols; ++k) {
        at[k] = nullptr;
        if (!c[k].host) continue;
        char *v = (char *)device_view(c[k].pinned ? c[k].host : so + c[k].at);
        if (!v) return false;
        at[k] = v + (size_t)(c[k].pinned ? g0 : c0) * c[k].row;
    }
    return true;
}

// Small batches (a MADS poll set): one stream, pinned scratch, one synchronisation.
#ifndef COV_ZC_IN_LIMIT
#define COV_ZC_IN_LIMIT (256u << 10) // the whole small-batch path; measured against 32 KiB: 512 candidates 53 -> 42 us, 2184 candidates 74 -> 62 us
#endif
#ifndef COV_ZC_MID_LIMIT
// measured on B200 (5 UAVs, pinned buffers, tools/batch_size_sweep.py): 4096 candidates 70 -> 55 us, 32 768 168 -> 133 us,
// 131 072 465 -> 392 us, 262 144 761 -> 715 us; level with the copy-engine pipeline at 524 288 (SM reads reach
// ~49 GB/s over PCIe, the DMA engine 55 GB/s), behind it at 1 M
#define COV_ZC_MID_LIMIT (48u << 20)
#endif
static int eval_host_small(cov_handle *h, const double *X, int64_t B, Cols &c, bool timed = true)
{
    const size_t in_bytes = (size_t)B * 3 * h->o.N * 8;
    const size_t out_bytes = pack_cols(c, (size_t)B);
    OK(ensure_pinned(h, &h->h_poll, &h->h_poll_cap, kPollBytes));
    char *hin = (char *)h->h_poll, *hout = (char *)h->h_poll + kPollOut;
    memcpy(hin, X, in_bytes);
    // poll-sized calls (a MADS poll set, the scalar closure): no copy engines at all -- the kernel reads the
    // candidates from the pinned scratch and writes the results into it over PCIe; the stream synchronise is
    // the only wait.  Saves two DMA set-ups per call, which is most of what a poll costs.
    char *vin = h->zero_copy_out && in_bytes <= (COV_ZC_IN_LIMIT) ? (char *)device_view(hin) : nullptr;
    char *vout = vin ? (char *)device_view(hout) : nullptr;
    const bool zc = vin && vout;
    if (!zc) {
        OK(ensure(h, h->dX, std::max<size_t>(in_bytes, 1 << 20)));
        OK(ensure(h, h->d_obj, std::max<size_t>(out_bytes, 1 << 20))); // one device block for every output
        CK(cudaMemcpyAsync(h->dX.p, hin, in_bytes, cudaMemcpyHostToDevice, h->stream));
    }
    char *base = zc ? vout : (char *)h->d_obj.p;
    char *at[kCols];
    for (int k = 0; k < kCols; ++k) at[k] = c[k].host ? base + c[k].at : nullptr;
    OK(launch_on_main(h, zc ? (const double *)vin : (const double *)h->dX.p, B, eval_out(at), timed));
    if (!zc) CK(cudaMemcpyAsync(hout, base, out_bytes, cudaMemcpyDeviceToHost, h->stream)); // ONE copy back
    CK(cudaStreamSynchronize(h->stream));
    for (const Col &col : c)
        if (col.host) memcpy(col.host, hout + col.at, (size_t)B * col.row);
    return COV_OK;
}

// Packed candidates (cov_eval_batch_packed): `elem`-byte values that the device widens to doubles, value * g.
struct PackedIn {
    const void *Q;
    int pack;
    double g;
    size_t elem;
};
static void unpack_host(const PackedIn &pk, size_t n, double *out) // the same arithmetic as unpack_kernel, for poll sets
{
    switch (pk.pack) {
    case COV_PACK_F32:
        for (size_t k = 0; k < n; ++k) out[k] = (double)((const float *)pk.Q)[k];
        break;
    case COV_PACK_I32:
        for (size_t k = 0; k < n; ++k) out[k] = (double)((const int32_t *)pk.Q)[k] * pk.g;
        break;
    default:
        for (size_t k = 0; k < n; ++k) out[k] = (double)((const int16_t *)pk.Q)[k] * pk.g;
        break;
    }
}

// best: the poll winner too (cov_argmin, cov_eval_batch_best), reduced on the device from the device-resident copy of
// the objectives and flags; 16 bytes come back per window.
static int eval_host(cov_handle *h, const double *X, int64_t B, double *obj, int64_t *count, uint8_t *feasible,
                     int64_t *class_count, double *progressive, Winner *best = nullptr, int barrier = 0,
                     const PackedIn *pk = nullptr)
{
    OK(check_ready(h, "cov_eval_batch"));
    if (B < 0 || (B > 0 && ((pk ? !pk->Q : !X) || (!obj && !best))))
        return fail(h, COV_ERR_INVALID, "cov_eval_batch: bad arguments");
    if (progressive && h->o.prog_which > h->o.N)
        return fail(h, COV_ERR_INVALID, "cov_eval_batch_ex: COV_OPT_PROGRESSIVE_INDEX names UAV " +
                                            std::to_string(h->o.prog_which) + " but N = " + std::to_string(h->o.N));
    if (B == 0) return COV_OK;
    recycle_spans(h);
    const int N = h->o.N;
    const int ncls = h->g.n_classes;
    const size_t row_bytes = (size_t)3 * N * 8;
    Cols c = {{(char *)obj, 8, &h->d_obj},
              {(char *)count, 8, &h->d_count},
              {(char *)class_count, (size_t)8 * ncls, &h->d_clscnt},
              {(char *)progressive, 8, &h->d_prog},
              {(char *)feasible, 1, &h->d_feas}};
    if (!best && (size_t)B * row_bytes <= (256u << 10) && (size_t)B * (25 + 8 * (size_t)ncls) <= (1536u << 10) && h->chunk == 0) {
        if (!pk) return eval_host_small(h, X, B, c);
        std::vector<double> wide((size_t)B * 3 * N); // a poll set: widened on the host, then the poll path as it is
        unpack_host(*pk, wide.size(), wide.data());
        return eval_host_small(h, wide.data(), B, c);
    }
    for (Col &col : c) col.pinned = !col.host || is_pinned_host(col.host);
#if COV_ZC_MID_LIMIT > 0
    // mid-size batches in pinned buffers: one launch that reads the candidates straight over PCIe (the
    // kernel's own unit prefetch overlaps transfer and compute) and writes the results back the same way
    if (!pk && !best && h->zero_copy_out && h->chunk == 0 && N <= 8 && (size_t)B * row_bytes <= (size_t)(COV_ZC_MID_LIMIT) && is_pinned_host(X) &&
        std::all_of(c, c + kCols, [](const Col &col) { return col.pinned; })) {
        const double *vx = (const double *)device_view((void *)X);
        char *at[kCols];
        if (vx && view_cols(c, nullptr, 0, 0, at)) {
            OK(launch_on_main(h, vx, B, eval_out(at), true));
            CK(cudaStreamSynchronize(h->stream));
            return COV_OK;
        }
    }
#endif
    // device window: at most ~1 GiB of candidates at a time
    const int64_t window = window_rows(B, row_bytes, 1ull << 30);
    // slice size: ~16 MiB of candidates, a multiple of 32 candidates (keeps device slices 16-byte aligned).
    // Packed input is compute-bound, not PCIe-bound (5 UAVs, int16: 0.54 ms of copies beside 0.7 ms of kernels per
    // 1 M candidates), so fewer, larger slices win: ~32 MiB of widened candidates (measured on B200, 1 M x 5 UAVs:
    // int16 1.126 -> 1.098 ms per call, int32 / float32 1.51 -> 1.37 ms; tools/packed_exp.py)
    const size_t slice_bytes = pk ? (32ull << 20) : (16ull << 20);
    int64_t chunk = h->chunk > 0 ? h->chunk : std::max<int64_t>(1024, (int64_t)(slice_bytes / row_bytes) / 32 * 32);
    chunk = std::min(chunk, window);
    // (two experiments lost here, DESIGN.md 5: a quarter- and a half-size first slice so that the kernels start sooner,
    // 1.107 -> 1.125 ms; and no copy engine at all, the widening kernel reading the pinned buffer over PCIe beside the
    // previous slice's objective kernel, 1.107 -> 1.21 ms)
    // the device columns: every requested one, obj always (the winner's input, or its mirror), feasible with best
    auto on_device = [&](int k) { return c[k].host || k == COL_OBJ || (k == COL_FEAS && best); };
    OK(ensure(h, h->dX, (size_t)window * row_bytes));
    for (int k = 0; k < kCols; ++k)
        if (on_device(k)) OK(ensure(h, *c[k].dev, (size_t)window * c[k].row));
    // what crosses PCIe per candidate: the doubles themselves, or the packed values (widened on the device)
    const size_t in_row_bytes = pk ? (size_t)3 * N * pk->elem : row_bytes;
    const char *in_base = pk ? (const char *)pk->Q : (const char *)X;
    const bool in_pinned = is_pinned_host(in_base);
    if (!in_pinned)
        for (int k = 0; k < 2; ++k) {
            size_t cap = h->h_in_cap;
            OK(ensure_pinned(h, &h->h_in[k], &cap, (size_t)chunk * in_row_bytes));
            if (k == 1) h->h_in_cap = cap;
        }
    if (pk)
        for (int k = 0; k < 2; ++k) OK(ensure(h, h->d_raw[k], (size_t)chunk * in_row_bytes));
    // outputs that are not pinned are staged per window and copied out at the window's end
    const size_t stage_out = pack_cols(c, (size_t)window);
    if (stage_out) OK(ensure_pinned(h, &h->h_out, &h->h_out_cap, stage_out));
    char *so = (char *)h->h_out;

    cudaEvent_t ev_in = get_event(h), ev_k = get_event(h), ev_free[2] = {get_event(h), get_event(h)};
    cudaEvent_t ev_raw[2] = {get_event(h), get_event(h)}; // packed input: slot k of d_raw has been widened
    bool free_armed[2] = {false, false}, raw_armed[2] = {false, false};
    int rc = COV_OK;
    auto done = [&](int code) {
        for (cudaEvent_t e : {ev_in, ev_k, ev_free[0], ev_free[1], ev_raw[0], ev_raw[1]}) h->ev_pool.push_back(e);
        return code;
    };
#define CKD(call)                                                         \
    do {                                                                  \
        cudaError_t e_ = (call);                                          \
        if (e_ != cudaSuccess) return done(fail_cuda(h, e_, #call));      \
    } while (0)
    // the copy streams must not start before earlier work on the main stream (grid/params) is done
    CKD(cudaEventRecord(ev_k, h->stream));
    CKD(cudaStreamWaitEvent(h->s_in, ev_k, 0));
    auto tr = [&](cudaStream_t s) {
        if (!h->trace) return;
        cudaEvent_t e = nullptr;
        cudaEventCreate(&e);
        cudaEventRecord(e, s);
        h->trace_ev.push_back(e);
    };
    for (cudaEvent_t e : h->trace_ev) cudaEventDestroy(e);
    h->trace_ev.clear();
    h->trace_ms.clear();
    tr(h->s_in);
    for (int64_t w0 = 0; w0 < B; w0 += window) {
        const int64_t wn = std::min(window, B - w0);
        int slot = 0;
        int64_t cn = 0;
        for (int64_t c0 = 0; c0 < wn; c0 += cn, slot ^= 1) {
            const int64_t left = wn - c0;
            cn = std::min(chunk, left);
            const char *src = in_base + (size_t)(w0 + c0) * in_row_bytes;
            double *dst = (double *)h->dX.p + (size_t)c0 * 3 * N;
            if (!in_pinned) {
                if (free_armed[slot]) CKD(cudaEventSynchronize(ev_free[slot]));
                host_copy(h, h->h_in[slot], src, (size_t)cn * in_row_bytes);
                src = (const char *)h->h_in[slot];
            }
            if (pk && raw_armed[slot]) CKD(cudaStreamWaitEvent(h->s_in, ev_raw[slot], 0)); // slot widened: reusable
            CKD(cudaMemcpyAsync(pk ? h->d_raw[slot].p : (void *)dst, src, (size_t)cn * in_row_bytes, cudaMemcpyHostToDevice,
                                h->s_in));
            if (!in_pinned) {
                CKD(cudaEventRecord(ev_free[slot], h->s_in));
                free_armed[slot] = true;
            }
            CKD(cudaEventRecord(ev_in, h->s_in));
            tr(h->s_in);
            CKD(cudaStreamWaitEvent(h->stream, ev_in, 0));
            tr(h->stream);
            if (pk) {
                CKD(launch_unpack(h->d_raw[slot].p, pk->pack, pk->g, dst, (long long)cn * 3 * N, h->stream));
                h->launches += 1;
                CKD(cudaEventRecord(ev_raw[slot], h->stream));
                raw_armed[slot] = true;
            }
            const int64_t g0 = w0 + c0;
            // results straight to pinned host memory (the caller's buffer, or the staging block): posted PCIe writes
            // of 17 B per candidate instead of three D2H copies per slice beside the H2D stream.  Not when a buffer is
            // one the device cannot address, nor for cov_argmin, which has no per-candidate outputs.
            char *at[kCols];
            const bool zc = h->zero_copy_out != 0 && (obj != nullptr || !best) && view_cols(c, so, g0, c0, at);
            if (!zc)
                for (int k = 0; k < kCols; ++k)
                    at[k] = on_device(k) ? (char *)c[k].dev->p + (size_t)c0 * c[k].row : nullptr;
            EvalOut out = eval_out(at);
            if (zc && best) { // results straight to the host as usual; the winner is reduced from device mirrors
                out.obj_mirror = (double *)h->d_obj.p + c0;
                out.feasible_mirror = (unsigned char *)h->d_feas.p + c0;
            }
            rc = launch_on_main(h, dst, cn, out, true);
            if (rc != COV_OK) return done(rc);
            CKD(cudaEventRecord(ev_k, h->stream));
            tr(h->stream);
            if (!zc) {
                CKD(cudaStreamWaitEvent(h->s_out, ev_k, 0));
                for (int k : {COL_OBJ, COL_COUNT, COL_FEAS, COL_CLS, COL_PROG}) {
                    const Col &col = c[k];
                    if (col.host)
                        CKD(cudaMemcpyAsync(col.pinned ? col.host + (size_t)g0 * col.row : so + col.at + (size_t)c0 * col.row,
                                            at[k], (size_t)cn * col.row, cudaMemcpyDeviceToHost, h->s_out));
                }
            }
            tr(zc ? h->stream : h->s_out);
        }
        // end of window: results home, device window reusable
        if (best && (rc = enqueue_winner(h, (const double *)h->d_obj.p, (const unsigned char *)h->d_feas.p, wn, barrier)) != COV_OK)
            return done(rc);
        CKD(cudaStreamSynchronize(h->stream));
        CKD(cudaStreamSynchronize(h->s_out));
        if (best) best->offer(h->h_small->win_obj, h->h_small->win_idx, w0);
        for (const Col &col : c)
            if (!col.pinned) host_copy(h, col.host + (size_t)w0 * col.row, so + col.at, (size_t)wn * col.row);
    }
#undef CKD
    if (h->trace && h->trace_ev.size() > 1) {
        for (size_t k = 1; k < h->trace_ev.size(); ++k) {
            float t = 0;
            cudaEventElapsedTime(&t, h->trace_ev[0], h->trace_ev[k]);
            h->trace_ms.push_back(t);
        }
    }
    return done(COV_OK);
}

extern "C" int cov_eval_batch_ex(cov_handle *h, const double *X, int64_t B, double *obj, int64_t *count,
                                 uint8_t *feasible, int64_t *class_count, double *progressive)
{
    if (!h) return fail(nullptr, COV_ERR_INVALID, "NULL handle");
    DeviceGuard dg(h->device);
    return eval_host(h, X, B, obj, count, feasible, class_count, progressive);
}

extern "C" int cov_eval_batch(cov_handle *h, const double *X, int64_t B, double *obj, int64_t *count,
                              uint8_t *feasible)
{
    return cov_eval_batch_ex(h, X, B, obj, count, feasible, nullptr, nullptr);
}

extern "C" int cov_eval_batch_best(cov_handle *h, const double *X, int64_t B, double *obj, int64_t *count,
                                   uint8_t *feasible, int32_t barrier, double *best_obj, int64_t *best_idx)
{
    if (!h) return fail(nullptr, COV_ERR_INVALID, "NULL handle");
    DeviceGuard dg(h->device);
    if (!best_obj || !best_idx) return fail(h, COV_ERR_INVALID, "cov_eval_batch_best: NULL winner outputs");
    Winner w;
    OK(eval_host(h, X, B, obj, count, feasible, nullptr, nullptr, &w, barrier));
    *best_obj = w.obj;
    *best_idx = w.idx;
    return COV_OK;
}

extern "C" int cov_eval_batch_packed(cov_handle *h, const void *Q, int32_t pack, double granularity, int64_t B, double *obj,
                                     int64_t *count, uint8_t *feasible, int32_t barrier, double *best_obj,
                                     int64_t *best_idx)
{
    if (!h) return fail(nullptr, COV_ERR_INVALID, "NULL handle");
    DeviceGuard dg(h->device);
    const size_t elem = pack == COV_PACK_F32 || pack == COV_PACK_I32 ? 4 : pack == COV_PACK_I16 ? 2 : 0;
    if (!elem) return fail(h, COV_ERR_INVALID, "cov_eval_batch_packed: pack must be COV_PACK_F32, _I32 or _I16");
    if (pack != COV_PACK_F32 && !(granularity > 0 && std::isfinite(granularity)))
        return fail(h, COV_ERR_INVALID, "cov_eval_batch_packed: granularity must be a positive finite number");
    if ((best_obj == nullptr) != (best_idx == nullptr))
        return fail(h, COV_ERR_INVALID, "cov_eval_batch_packed: best_obj and best_idx go together");
    PackedIn pk{Q, pack, granularity, elem};
    if (!best_obj) return eval_host(h, nullptr, B, obj, count, feasible, nullptr, nullptr, nullptr, 0, &pk);
    Winner w;
    OK(eval_host(h, nullptr, B, obj, count, feasible, nullptr, nullptr, &w, barrier, &pk));
    *best_obj = w.obj;
    *best_idx = w.idx;
    return COV_OK;
}

// One candidate through the small path, its launch untimed: copy in, one launch, copy out, one synchronisation.
extern "C" int cov_eval_one(cov_handle *h, const double *x, double *obj)
{
    if (!h) return fail(nullptr, COV_ERR_INVALID, "NULL handle");
    DeviceGuard dg(h->device);
    OK(check_ready(h, "cov_eval_one"));
    if (!x || !obj) return fail(h, COV_ERR_INVALID, "cov_eval_one: NULL argument");
    recycle_spans(h);
    Cols c = {{(char *)obj, 8, &h->d_obj}}; // the objective alone
    return eval_host_small(h, x, 1, c, false);
}


// ------------------------------------------------------------------------------------------
// the batched MADS poll driver in native code (SURVEY.md 8f-1): the caller of the objective.
// Same settings as the reference's TDM_STATIC_opt.optimize (src/TDM_STATIC_opt.jl:118-222: iteration
// limit, granularity on every variable, extreme barrier from the fused constraints, feasible incumbent
// else the start point) and the same published algorithm as mads.py (granular mesh of Audet, Le Digabel &
// Tribes 2019: poll size a * 10^b with a in {1, 2, 5}, mesh size max(10^(b - |b - b0|), granularity),
// 2n directions from a random Householder matrix rounded onto the mesh, complete polling); every poll
// set is ONE launch through the small-batch path.  DirectSearch.jl's own iterates are not reproducible
// (unseeded LTMADS), so trajectories are not a parity target; objective values are.
// ------------------------------------------------------------------------------------------
namespace {
struct Rng { // splitmix64 + Box-Muller: self-contained, seedable
    uint64_t s;
    uint64_t next()
    {
        uint64_t z = (s += 0x9E3779B97F4A7C15ull);
        z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
        z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
        return z ^ (z >> 31);
    }
    double u01() { return ((double)(next() >> 11) + 0.5) * (1.0 / 9007199254740992.0); }
    double normal() { return std::sqrt(-2.0 * std::log(u01())) * std::cos(6.283185307179586 * u01()); }
};
struct MeshVar {
    double a;
    int b, b0;
};
// initial poll size: about |x0_i| / 10 (at least 1), on the {1, 2, 5} x 10^b ladder.  A non-finite start keeps the
// conversion defined: +-Inf gets b = -kMadsPow10Min (the device's powers-of-ten table clamps there too), NaN gets b = 0
// (target >= 1 otherwise, so b >= 0); either way a = 5, as the mantissa is NaN.
MeshVar initial_mesh(double x0, double g)
{
    const double target = std::max(std::max(std::fabs(x0) / 10.0, 1.0), g);
    const double lb = std::floor(std::log10(target));
    const int b = lb == lb ? (int)std::min(lb, (double)-kMadsPow10Min) : 0;
    const double mant = target / std::pow(10.0, b);
    return {mant < 2 ? 1.0 : (mant < 5 ? 2.0 : 5.0), b, b};
}
} // namespace

extern "C" int cov_mads_solve(cov_handle *h, const double *x0, int64_t n_iter, double granularity, uint64_t seed,
                              double *x_out, double *obj_out, int64_t *stats)
{
    if (!h) return fail(nullptr, COV_ERR_INVALID, "NULL handle");
    DeviceGuard dg(h->device);
    OK(check_ready(h, "cov_mads_solve"));
    if (!x0 || !x_out || n_iter < 0 || !(granularity >= 0)) return fail(h, COV_ERR_INVALID, "cov_mads_solve: bad arguments");
    const int n = 3 * h->o.N;
    const double g = granularity;
    auto snap = [g](double v) { return g > 0 ? std::nearbyint(v / g) * g : v; };
    std::unordered_map<std::string, double> cache;
    int64_t evaluations = 0, batches = 0, successes = 0, iterations = 0;
    std::vector<double> P, vals;
    std::vector<uint8_t> feas;
    auto key_of = [n](const double *p) { return std::string(reinterpret_cast<const char *>(p), (size_t)n * 8); };
    // objective with the extreme barrier for the rows of P that are not cached yet
    auto evaluate = [&](const std::vector<double> &pts, std::vector<double> &f) -> int {
        const int64_t m = (int64_t)pts.size() / n;
        f.assign((size_t)m, 0.0);
        std::vector<int64_t> todo;
        std::vector<double> Q;
        for (int64_t k = 0; k < m; ++k) {
            auto it = cache.find(key_of(&pts[(size_t)k * n]));
            if (it != cache.end()) f[(size_t)k] = it->second;
            else {
                todo.push_back(k);
                Q.insert(Q.end(), &pts[(size_t)k * n], &pts[(size_t)k * n] + n);
            }
        }
        if (!todo.empty()) {
            vals.assign(todo.size(), 0.0);
            feas.assign(todo.size(), 1);
            recycle_spans(h);
            OK(eval_host(h, Q.data(), (int64_t)todo.size(), vals.data(), nullptr, feas.data(), nullptr, nullptr));
            evaluations += (int64_t)todo.size();
            batches += 1;
            for (size_t q = 0; q < todo.size(); ++q) {
                const double v = (feas[q] && vals[q] == vals[q]) ? vals[q] : INFINITY;
                cache[key_of(&Q[q * n])] = v;
                f[(size_t)todo[q]] = v;
            }
        }
        return COV_OK;
    };
    std::vector<double> x(x0, x0 + n), f;
    OK(evaluate(x, f));
    double fx = f[0];
    bool feasible_found = std::isfinite(fx);
    std::vector<MeshVar> mesh((size_t)n);
    for (int i = 0; i < n; ++i) mesh[i] = initial_mesh(x[i], g);
    Rng rng{seed * 0x9E3779B97F4A7C15ull + 0x1234567ull};
    std::vector<double> v((size_t)n), H((size_t)n * n), delta((size_t)n), rho((size_t)n);
    for (int64_t it = 0; it < n_iter; ++it) {
        ++iterations;
        for (int i = 0; i < n; ++i) {
            const double Delta = std::max(mesh[i].a * std::pow(10.0, mesh[i].b), g);
            delta[i] = std::max(std::pow(10.0, mesh[i].b - std::abs(mesh[i].b - mesh[i].b0)), g);
            rho[i] = std::max(std::nearbyint(Delta / delta[i]), 1.0);
        }
        double nrm = 0;
        for (int i = 0; i < n; ++i) {
            v[i] = rng.normal();
            nrm += v[i] * v[i];
        }
        nrm = std::sqrt(nrm);
        for (int i = 0; i < n; ++i) v[i] /= nrm;
        P.clear();
        for (int sgn = 1; sgn >= -1; sgn -= 2)
            for (int j = 0; j < n; ++j) { // column j of I - 2 v v^T, scaled to the poll-to-mesh ratio, rounded
                double hmax = 0;
                for (int i = 0; i < n; ++i) {
                    H[i] = (i == j ? 1.0 : 0.0) - 2.0 * v[i] * v[j];
                    hmax = std::max(hmax, std::fabs(H[i]));
                }
                bool any = false, moved = false;
                const size_t at = P.size();
                P.resize(at + n);
                for (int i = 0; i < n; ++i) {
                    const double d = std::nearbyint(rho[i] * H[i] / hmax);
                    any |= d != 0;
                    P[at + i] = snap(x[i] + sgn * d * delta[i]);
                    moved |= P[at + i] != x[i];
                }
                if (!any || !moved) P.resize(at);
            }
        // drop exact duplicates (keep the first)
        {
            std::unordered_map<std::string, int> seen;
            std::vector<double> U;
            for (size_t k = 0; k * n < P.size(); ++k)
                if (seen.emplace(key_of(&P[k * n]), 1).second) U.insert(U.end(), &P[k * n], &P[k * n] + n);
            P.swap(U);
        }
        double best = INFINITY;
        size_t kb = 0;
        if (!P.empty()) {
            OK(evaluate(P, f));
            for (size_t k = 0; k < f.size(); ++k)
                if (f[k] < best) {
                    best = f[k];
                    kb = k;
                }
        }
        if (best < fx || (!feasible_found && std::isfinite(best))) {
            std::copy(&P[kb * n], &P[kb * n] + n, x.begin());
            fx = best;
            feasible_found = true;
            ++successes;
            for (auto &m : mesh) { // enlarge
                if (m.a == 1.0) m.a = 2.0;
                else if (m.a == 2.0) m.a = 5.0;
                else {
                    m.a = 1.0;
                    ++m.b;
                }
            }
        } else { // refine; stop when every poll size sits at its granularity
            bool moved = false;
            for (auto &m : mesh) {
                if (g > 0 && m.a * std::pow(10.0, m.b) <= g) continue;
                if (m.a == 1.0) {
                    m.a = 5.0;
                    --m.b;
                } else if (m.a == 2.0) m.a = 1.0;
                else m.a = 2.0;
                moved = true;
            }
            if (!moved) break;
        }
    }
    const double *res = feasible_found ? x.data() : x0; // p.x if a feasible incumbent exists, else the start (p.i)
    std::copy(res, res + n, x_out);
    if (obj_out) *obj_out = fx;
    if (stats) {
        stats[0] = iterations;
        stats[1] = evaluations;
        stats[2] = batches;
        stats[3] = successes;
    }
    return COV_OK;
}

// The solver's launch plan: N <= kMadsMaxUavs and, with the cell store's objective (grid: its description, NULL for
// the region objective), one warp's framebuffer.
static int check_mads_limits(cov_handle *h, const char *who, const GridDesc *grid)
{
    const int N = h->o.N;
    int warps = 0, smem = 0, planes_smem = 0;
    if (N > kMadsMaxUavs)
        return fail(h, COV_ERR_LIMIT, std::string(who) + ": N = " + std::to_string(N) + " exceeds the " +
                                          std::to_string(kMadsMaxUavs) + " UAVs of the solver's launch plan");
    if (grid && !mads_plan(*grid, N, h->cfg, &warps, &smem, &planes_smem))
        return fail(h, COV_ERR_LIMIT, std::string(who) + ": one warp's framebuffer of the " +
                                          std::to_string(h->g.nx) + " x " + std::to_string(h->g.ny) +
                                          " grid does not fit the " + std::to_string(h->cfg.max_smem_optin) +
                                          " bytes of shared memory per CTA");
    return COV_OK;
}

constexpr size_t kPow10Bytes = (1 - 2 * kMadsPow10Min) * 8;
// The device buffers of S solves of n variables, allocated and pointed at by a: mads_in = [prefix, which opens with the
// powers of ten from the host's libm | X0: S n doubles | a0: S n doubles | b0: S n ints], mads_out = [X_out: S n doubles |
// obj: S | stats: S x 4 | extra_out bytes].  Fills pow10 into hin, the host copy of mads_in (at least prefix bytes).
static int mads_buffers(cov_handle *h, size_t prefix, int64_t S, int n, size_t extra_out, std::vector<unsigned char> &hin,
                        MadsArgs &a)
{
    const size_t sn = (size_t)S * n;
    OK(ensure(h, h->mads_in, prefix + sn * 20));
    OK(ensure(h, h->mads_out, sn * 8 + (size_t)S * 40 + extra_out));
    for (int b = kMadsPow10Min; b <= -kMadsPow10Min; ++b) ((double *)hin.data())[b - kMadsPow10Min] = std::pow(10.0, b);
    a = MadsArgs{};
    a.pow10 = (const double *)h->mads_in.p;
    a.X0 = (const double *)((const char *)h->mads_in.p + prefix);
    a.a0 = a.X0 + sn;
    a.b0 = (const int *)(a.a0 + sn);
    a.X_out = (double *)h->mads_out.p;
    a.obj_out = a.X_out + sn;
    a.stats = (long long *)(a.obj_out + S);
    a.S = S;
    a.force_exact = h->cfg.force_exact;
    return COV_OK;
}

// S solves of the same loop on the device, one launch for all of them (cov_mads.cu).  The host contributes what
// must carry its libm's bits: the initial mesh of every start and the table of powers of ten.  region: the objective
// of cov_eval_region_batch instead of the cell store's.
static int mads_solve_batch(cov_handle *h, bool region, const double *X0, int64_t S, int64_t n_iter, double granularity,
                            uint64_t seed, double *X_out, double *obj_out, int64_t *stats)
{
    const char *who = region ? "cov_mads_solve_batch_region" : "cov_mads_solve_batch";
    if (S < 0 || n_iter < 0 || !(granularity >= 0) || (S > 0 && (!X0 || !X_out)))
        return fail(h, COV_ERR_INVALID, std::string(who) + ": bad arguments");
    if (S == 0) return COV_OK;
    const int N = h->o.N, n = 3 * N;
    OK(check_mads_limits(h, who, region ? nullptr : &h->g));
    if (!region && !h->area_exact) OK(entries_on_device(h)); // non-dyadic weights: the list-order sum
    const size_t sn = (size_t)S * n, in_bytes = kPow10Bytes + sn * 20, out_bytes = sn * 8 + (size_t)S * 40;
    std::vector<unsigned char> hin(in_bytes), hout(out_bytes);
    MadsArgs a;
    OK(mads_buffers(h, kPow10Bytes, S, n, 0, hin, a)); // the prefix: pow10
    double *hx = (double *)(hin.data() + kPow10Bytes), *ha = hx + sn;
    int *hb = (int *)(ha + sn);
    memcpy(hx, X0, sn * 8);
    for (size_t q = 0; q < sn; ++q) {
        const MeshVar m = initial_mesh(X0[q], granularity);
        ha[q] = m.a;
        hb[q] = m.b;
    }
    unsigned char *din = (unsigned char *)h->mads_in.p, *dout = (unsigned char *)h->mads_out.p;
    CK(cudaMemcpyAsync(din, hin.data(), in_bytes, cudaMemcpyHostToDevice, h->stream));
    a.n_iter = n_iter;
    a.granularity = granularity;
    a.seed = seed;
    a.ordered = h->area_exact ? 0 : 1;
    unsigned long long *counter = nullptr;
    OK(take_counter(h, &counter));
    cudaError_t e = region ? launch_mads_region(h->region, h->o, h->cfg, a, counter, h->stream)
                           : launch_mads(h->g, h->o, h->cfg, a, counter, h->stream);
    if (e != cudaSuccess) return fail_cuda(h, e, (std::string(who) + ": kernel launch").c_str());
    h->launches += 1;
    CK(cudaMemcpyAsync(hout.data(), dout, out_bytes, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    memcpy(X_out, hout.data(), sn * 8);
    if (obj_out) memcpy(obj_out, hout.data() + sn * 8, (size_t)S * 8);
    if (stats) memcpy(stats, hout.data() + sn * 8 + (size_t)S * 8, (size_t)S * 4 * 8);
    return COV_OK;
}

extern "C" int cov_mads_solve_batch(cov_handle *h, const double *X0, int64_t S, int64_t n_iter, double granularity,
                                    uint64_t seed, double *X_out, double *obj_out, int64_t *stats)
{
    if (!h) return fail(nullptr, COV_ERR_INVALID, "NULL handle");
    DeviceGuard dg(h->device);
    OK(check_ready(h, "cov_mads_solve_batch"));
    return mads_solve_batch(h, false, X0, S, n_iter, granularity, seed, X_out, obj_out, stats);
}

// The append step that opens every timestep of a dynamic horizon (run_horizon; NULL: the static loop).  g is the
// store's envelope: a plane set that holds every multiplicity the loop can reach, fixed for the whole loop.  An empty
// plane adds nothing to any count, so every objective value is the one of the smaller plane set the host path has.
struct HorizonAppend {
    GridDesc g{};
    int n_classes = 0; // the classes after the call: the store's, then the new weights in order of first appearance
    double cw[kMaxClasses] = {0, 0, 0, 0};
    // the fire list (cov_run_horizon_points): timestep t appends entries offsets[t-1] .. offsets[t]-1 of (cell, pcls);
    // with list_of (cov_run_horizon_points_ensemble, E values in [0, L)), scenario e follows schedule l = list_of[e]:
    // entries offsets[l*T + t-1] .. offsets[l*T + t]-1
    const int64_t *offsets = nullptr;
    const int64_t *list_of = nullptr;
    int64_t L = 1;
    std::vector<int> cell;
    std::vector<unsigned char> pcls;
    bool stamps = false; // record the last timestep that removed entries from each cell
    // the automaton (cov_run_horizon_fire): fire_steps[t-1] steps with append at timestep t, numbered from first_step,
    // with scenario e's 9 direction probabilities at fire_p + 9e (host) and its key fire_seed + e * fire_seed_stride
    const int64_t *fire_steps = nullptr;
    const double *fire_p = nullptr;
    uint64_t fire_seed = 0, fire_seed_stride = 0;
    int64_t first_step = 0;
};

// The arguments every horizon call takes (the last of cov_run_horizon's checks).
static int check_horizon_args(cov_handle *h, const char *who, const double *x_start, int64_t T, int64_t S, double spread,
                              int64_t n_iter, double granularity, const double *boxes, int64_t n_boxes,
                              const double *X_out)
{
    if (T < 0 || S < 1 || n_iter < 0 || (T > 0 && (!x_start || !X_out)) || !std::isfinite(spread) || spread < 0 ||
        !(granularity >= 0) || n_boxes < 0 || (n_boxes > 0 && !boxes))
        return fail(h, COV_ERR_INVALID, std::string(who) + ": bad arguments");
    return COV_OK;
}

// The arguments and store every horizon call needs (cov_run_horizon's checks, in its order).  list_ok: the call can
// replay the list-order sum (not the automaton), which it does when COV_OPT_LIST_ORDER_HORIZON is 1.
static int check_horizon(cov_handle *h, const char *who, const double *x_start, int64_t T, int64_t S, double spread,
                         int64_t n_iter, double granularity, const double *boxes, int64_t n_boxes, const double *X_out,
                         bool list_ok)
{
    OK(check_ready(h, who));
    if (!h->o.use_cons3)
        return fail(h, COV_ERR_STATE, std::string(who) + ": the parameters have no previous swarm (cons3 is off)");
    if (!h->area_exact && !(list_ok && h->list_order_horizon))
        return fail(h, COV_ERR_STATE, std::string(who) + ": the store's area depends on the list order (area_exact == 0)");
    return check_horizon_args(h, who, x_start, T, S, spread, n_iter, granularity, boxes, n_boxes, X_out);
}

// The envelope's plane set: for class k, planes for bits 0 .. floor(log2(max_mult[k])), where max_mult[k] bounds the
// multiplicity of every cell of class k over the whole loop; n_entries bounds the entries.  Removals are ignored, so
// the refusals are conservative.  list (NULL: refused, the automaton): whether the loop needs the list-order sum,
// accepted when COV_OPT_LIST_ORDER_HORIZON is 1.
static int horizon_envelope(cov_handle *h, const char *who, HorizonAppend &app, const unsigned *max_mult,
                            int64_t n_entries, bool *list)
{
    GridDesc &g = app.g;
    g = h->g;
    g.n_classes = app.n_classes;
    for (int k = 0; k < kMaxClasses; ++k) g.class_weight[k] = k < app.n_classes ? app.cw[k] : 0.0;
    int np = 0;
    for (int k = 0; k < g.n_classes; ++k)
        for (int b = 0; b < 8 && (max_mult[k] >> b); ++b) {
            if (np >= kMaxPlanes)
                return fail(h, COV_ERR_LIMIT, std::string(who) + ": the store can reach more than 8 bit planes "
                                                                 "(weight classes x multiplicity bits, removals ignored)");
            g.plane_class[np] = k;
            g.plane_mult[np] = 1 << b;
            ++np;
        }
    if (np == 0) { // an empty store: one all-zero plane, as rebuild_planes keeps it
        g.plane_class[0] = 0;
        g.plane_mult[0] = 1;
        np = 1;
    }
    for (int l = np; l < kMaxPlanes; ++l) {
        g.plane_class[l] = 0;
        g.plane_mult[l] = 0;
    }
    g.n_planes = np;
    g.planes = nullptr; // run_horizon points them at the handle's buffers
    g.planes_q = nullptr;
    const bool exact = sums_exact(g, n_entries);
    if (!exact && !(list && h->list_order_horizon))
        return fail(h, COV_ERR_STATE, std::string(who) + ": with every entry the call can add, the store's area "
                                                         "would depend on the list order (area_exact == 0)");
    if (list) *list = !exact;
    return check_mads_limits(h, who, &g);
}

// The list mirror after a fire-list horizon (the pending removals of the call's start already applied): an entry
// appended at timestep ta (ta = 1 for those in the list before the call) survives iff no timestep >= ta removed
// entries from its cell, i.e. iff stamp[cell] < ta.
static void entries_replay(cov_handle *h, const HorizonAppend &app, int64_t T, const int *stamp)
{
    size_t keep = 0;
    for (size_t p = 0; p < h->ent_cell_h.size(); ++p)
        if (stamp[h->ent_cell_h[p]] < 1) {
            h->ent_cell_h[keep] = h->ent_cell_h[p];
            h->ent_cls_h[keep] = h->ent_cls_h[p];
            ++keep;
        }
    h->ent_cell_h.resize(keep);
    h->ent_cls_h.resize(keep);
    for (int64_t t = 1; t <= T; ++t)
        for (int64_t q = app.offsets[t - 1]; q < app.offsets[t]; ++q)
            if (stamp[app.cell[(size_t)q]] < t) {
                h->ent_cell_h.push_back(app.cell[(size_t)q]);
                h->ent_cls_h.push_back(app.pcls[(size_t)q]);
            }
    h->ent_removed_pending = false;
    h->ent_dev_valid = false;
}

// The scenarios of cov_run_horizon_ensemble / cov_run_horizon_fire_ensemble / cov_run_horizon_points_ensemble
// (run_horizon; NULL: one scenario on the handle's own store): E copies of the handle's store, parameters and automaton
// state, made on the device when the call starts and dropped when it ends.
struct HorizonEnsemble {
    int64_t E = 1;
    uint8_t *cells_out = nullptr;  // E x nx*ny (nullable): the multiplicities each scenario leaves
    uint8_t *states_out = nullptr; // E x nx*ny (nullable): the automaton state each scenario leaves
};

// The scenario counts the ensemble calls accept: E * S solves per launch (counted in int by the grid and the
// dispenser), E * T * S keys without wrapping.
static int check_ensemble(cov_handle *h, const char *who, int64_t E, int64_t T, int64_t S)
{
    if (E < 1 || E > INT32_MAX / S || (T > 0 && E * S > INT64_MAX / T))
        return fail(h, COV_ERR_INVALID, std::string(who) + ": E must be >= 1 with E * S <= 2^31 - 1 and E * T * S <= "
                                                           "2^63 - 1");
    return COV_OK;
}

// The end of an ensemble call: a large ensemble would otherwise pin E copies of the store for the handle's lifetime.
static int drop_ensemble(cov_handle *h, int rc)
{
    if (h->ens.p) {
        (void)cudaStreamSynchronize(h->stream); // a failed call may still have copies in flight
        (void)cudaFree(h->ens.p);
        (void)cudaGetLastError();
        h->ens = DevBuf{};
    }
    return rc;
}

// E copies of `bytes` bytes at src side by side at dst (device memory), in 1 + ceil(log2(E)) copies.
static cudaError_t replicate(void *dst, const void *src, size_t bytes, int64_t E, cudaStream_t s)
{
    cudaError_t e = cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, s);
    for (int64_t have = 1; have < E && e == cudaSuccess; have *= 2)
        e = cudaMemcpyAsync((char *)dst + (size_t)have * bytes, dst, (size_t)std::min(have, E - have) * bytes,
                            cudaMemcpyDeviceToDevice, s);
    return e;
}

// T >= 1 timesteps of FullSimulation.py's MADS loop (lines 72-107) with S starts per timestep, all enqueued before the
// one synchronise at the end (arguments and solver limits checked by the caller).  Per timestep: the append step of
// app (update_POI's push! or the automaton), rmvCoveredPOI of cur into the stats row, the bit planes repacked (the
// plane set stays fixed: removals only clear multiplicities, and app's envelope holds every append), the r_max rule /
// cons3's previous swarm / the starts (horizon_start_kernel), S solves (launch_mads), the winner to cur
// (horizon_commit_kernel), AreaMaxObjective(cur).  stamps_out (nullable, nx*ny): app's removal stamps.
// ens: the same loop over ens->E scenarios side by side (one launch per step for all of them) on copies of the store
// and parameters (and, with the automaton, of its state); x_start and the outputs then hold E scenarios, each of them
// as the single call lays it out, and with the fire list each scenario appends its own schedule (app->list_of).
// list: the store's area depends on the list order (COV_OPT_LIST_ORDER_HORIZON): the solves and the objective walk
// each scenario's point list (ListWalk: the handle's list, then the schedule's entries, live by the removal stamps,
// which are then always kept), and nothing reads the bit planes, so they are not repacked.
static int run_horizon(cov_handle *h, const char *who, const double *x_start, int64_t T, int64_t S, double spread,
                       int64_t n_iter, double granularity, uint64_t seed, const double *boxes, int64_t n_boxes,
                       double h_focus, double h_max, double *X_out, double *obj_out, int64_t *stats, double *step_ms,
                       HorizonAppend *app, int *stamps_out, bool list, const HorizonEnsemble *ens = nullptr)
{
    if (list) OK(entries_on_device(h)); // the base list: the handle's, its pending removals applied
    GridDesc lg = app ? app->g : h->g;
    const int64_t E = ens ? ens->E : 1;
    const int N = h->o.N, n = 3 * N, cols = app ? 5 : 4;
    const size_t ncell = (size_t)h->g.nx * h->g.ny, P = app ? app->cell.size() : 0;
    const bool stamps = app && app->stamps, automaton = app && app->fire_steps;
    const int64_t *list_of = app ? app->list_of : nullptr;
    const bool walk_sched = list && app && app->offsets; // the list walk reads the schedules' offsets
    const size_t n_off = list_of || walk_sched ? (size_t)(app->L * T + 1) : 0;
    // in: [pow10 | x_start: E n | boxes: 4 n_boxes | direction probabilities: E 9 | the schedules' offsets: L T + 1 |
    // list_of: E | appended cells: P ints | their append timesteps (list): P ints | their classes: P bytes | the
    // solves' inputs]; out: [the solves' outputs | X_out: T E n | obj_out: T E | stats: T E cols | removal stamps: E nx*ny
    // ints (on the device, and downloaded with stamps)], timestep-major (a timestep's rows side by side); pinned: [the
    // out rows after the solves' | the cells: E nx*ny | the automaton states: E nx*ny]
    const size_t tn = (size_t)T * E * n;
    const size_t o_x = kPow10Bytes, o_box = o_x + (size_t)E * n * 8, o_fp = o_box + (size_t)n_boxes * 32;
    const size_t o_off = o_fp + (automaton ? (size_t)E * 9 * 8 : 0), o_list = o_off + n_off * 8;
    const size_t o_cell = o_list + (list_of ? (size_t)E * 8 : 0), o_ta = o_cell + P * 4;
    const size_t o_cls = o_ta + (list ? P * 4 : 0), o_X0 = (o_cls + P + 7) / 8 * 8;
    const size_t o_stamp = tn * 8 + (size_t)T * E * 8 + (size_t)T * E * cols * 8;
    const size_t res_bytes = o_stamp + (stamps ? (size_t)E * ncell * 4 : 0);
    const size_t dev_bytes = o_stamp + (stamps || list ? (size_t)E * ncell * 4 : 0);
    const size_t cells_bytes = ens && ens->cells_out ? (size_t)E * ncell : 0;
    const size_t states_bytes = ens && automaton && ens->states_out ? (size_t)E * ncell : 0;
    std::vector<unsigned char> hin(o_X0);
    MadsArgs a;
    OK(mads_buffers(h, o_X0, E * S, n, dev_bytes, hin, a));
    memcpy(hin.data() + o_x, x_start, (size_t)E * n * 8);
    if (n_boxes) memcpy(hin.data() + o_box, boxes, (size_t)n_boxes * 32);
    if (automaton) memcpy(hin.data() + o_fp, app->fire_p, (size_t)E * 9 * 8);
    if (n_off) memcpy(hin.data() + o_off, app->offsets, n_off * 8);
    if (list_of) memcpy(hin.data() + o_list, list_of, (size_t)E * 8);
    if (P) {
        memcpy(hin.data() + o_cell, app->cell.data(), P * 4);
        memcpy(hin.data() + o_cls, app->pcls.data(), P);
    }
    if (list && P) { // entry q of schedule l is appended at the t with offsets[l T + t-1] <= q < offsets[l T + t]
        int *ta = (int *)(hin.data() + o_ta);
        for (int64_t l = 0; l < app->L; ++l)
            for (int64_t t = 1; t <= T; ++t)
                for (int64_t q = app->offsets[l * T + t - 1]; q < app->offsets[l * T + t]; ++q) ta[q] = (int)t;
    }
    // the scenarios' device state: [mult: E nx*ny | cls: E nx*ny | automaton states: 2 E nx*ny, the E of either
    // ping-pong half side by side | plane sets: E | the single-plane swizzled copy, for E = 1 (launch_eval's CTA kernel
    // may read it; the E > 1 kernels read the packed planes) | parameters: E 5N | thresholds: E 3N]; cls, the states and
    // the plane sets from 16-byte boundaries: add_points_kernel's 32-bit atomics need 4-byte aligned bases for mult, cls
    const size_t pw = (size_t)lg.n_planes * lg.plane_words * 4, q_bytes = ((size_t)h->g.ny * h->g.qstride + 8) * 4;
    const bool quad = E == 1 && (app ? lg.n_planes == 1 : lg.planes_q != nullptr); // as the single call has it
    const size_t store16 = ((size_t)E * ncell + 15) / 16 * 16, o_efire = 2 * store16;
    const size_t o_epl = (o_efire + (automaton ? 2 * store16 : 0) + 15) / 16 * 16;
    const size_t o_eq = o_epl + (size_t)E * pw;
    const size_t o_epar = o_eq + (quad ? q_bytes : 0), o_exyT = o_epar + (size_t)E * 5 * N * 8;
    if (ens) OK(ensure(h, h->ens, o_exyT + (size_t)E * n * 8));
    else OK(ensure(h, h->xyT, (size_t)n * 8));
    OK(ensure_pinned(h, &h->h_out, &h->h_out_cap, res_bytes + cells_bytes + states_bytes));
    if (app && !ens) { // the envelope's planes; rebuild_planes sizes them for the store again at the end
        int rc = ensure(h, h->planes, (size_t)lg.n_planes * lg.plane_words * 4);
        if (rc == COV_OK && lg.n_planes == 1) rc = ensure(h, h->planes_q, q_bytes);
        if (rc != COV_OK) { // a buffer may have moved: describe the unchanged store again
            const std::string msg = h->err;
            if (rebuild_planes(h, h->g.n_classes, h->g.class_weight) != COV_OK) h->have_grid = false;
            h->err = msg;
            return rc;
        }
        lg.planes = (const uint32_t *)h->planes.p;
        lg.planes_q = lg.n_planes == 1 ? (const uint32_t *)h->planes_q.p : nullptr;
    }
    unsigned char *din = (unsigned char *)h->mads_in.p;
    const double *d_x0 = (const double *)(din + o_x);
    const int *d_cell = (const int *)(din + o_cell);
    const unsigned char *d_cls = din + o_cls;
    const double *d_fp = (const double *)(din + o_fp);
    const long long *d_off = (const long long *)(din + o_off), *d_list = (const long long *)(din + o_list);
    double *d_Xo = (double *)(a.stats + 4 * E * S), *d_oo = d_Xo + tn, *xyT = (double *)h->xyT.p;
    long long *d_st = (long long *)(d_oo + T * E);
    unsigned char *mult = (unsigned char *)h->mult.p, *cls = (unsigned char *)h->cls.p;
    double *params = (double *)h->params.p;
    unsigned char *fire[2] = {(unsigned char *)h->fire[0].p, (unsigned char *)h->fire[1].p};
    int fire_cur = h->fire_cur;
    ObjParams o = h->o;
    if (ens) {
        unsigned char *eb = (unsigned char *)h->ens.p;
        mult = eb;
        cls = eb + store16;
        fire[0] = eb + o_efire; // the scenarios start in half 0: one parity for all of them (the schedule is shared)
        fire[1] = fire[0] + store16;
        fire_cur = 0;
        lg.planes = (const uint32_t *)(eb + o_epl);
        lg.planes_q = quad ? (const uint32_t *)(eb + o_eq) : nullptr;
        params = (double *)(eb + o_epar);
        xyT = (double *)(eb + o_exyT);
        o.r_max = params; // scenario e's block at e * 5N (the kernels shift these by it)
        o.prev_x = params + N;
        o.prev_y = params + 2 * N;
        o.prev_z = params + 3 * N;
        o.cons3_G = params + 4 * N;
    }
    int *d_stamp = stamps || list ? (int *)((unsigned char *)d_Xo + o_stamp) : nullptr;
    ListWalk walk{};
    if (list) {
        walk.base_cell = h->g.ent_cell;
        walk.base_cls = h->g.ent_cls;
        walk.n_base = h->g.n_ent;
        walk.cell = d_cell;
        walk.cls = d_cls;
        walk.ta = (const int *)(din + o_ta);
        walk.off = walk_sched ? d_off : nullptr;
        walk.list_of = list_of ? d_list : nullptr;
        walk.T = T;
        walk.ncell = (long long)ncell;
        walk.stamps = d_stamp;
    }
    a.n_iter = n_iter;
    a.granularity = granularity;
    a.ordered = 0;
    HorizonStep hs{};
    hs.N = N;
    hs.n_boxes = (int)n_boxes;
    hs.S = S;
    hs.E = E;
    hs.spread = spread;
    hs.granularity = granularity;
    hs.seed = seed;
    hs.seed_stride = (uint64_t)T * (uint64_t)S;
    hs.pow10 = a.pow10;
    hs.boxes = (const double *)(din + o_box);
    hs.h_focus = h_focus;
    hs.h_max = h_max;
    hs.tan_half_fov = h->o.tan_half_fov;
    LaunchCfg cfg = h->cfg; // a dyadic store: every kernel gives the list-order sum, the stale device list is not needed
    cfg.ordered = 0;
    if (cfg.kernel == COV_KERNEL_ORDERED) cfg.kernel = COV_KERNEL_AUTO;
    int *overflow = (int *)h->overflow.p;
    int64_t step = app ? app->first_step : 0;
    std::vector<cudaEvent_t> ev;
    if (step_ms)
        for (int64_t t = 0; t <= T; ++t) ev.push_back(get_event(h));

    cudaError_t e = cudaMemcpyAsync(din, hin.data(), o_X0, cudaMemcpyHostToDevice, h->stream);
    const char *what = "upload";
    if (ens && e == cudaSuccess) { // the scenarios start from the handle's store and parameters
        what = "scenario copies";
        e = replicate(mult, h->mult.p, ncell, E, h->stream);
        if (e == cudaSuccess) e = replicate(cls, h->cls.p, ncell, E, h->stream);
        if (e == cudaSuccess) e = replicate(params, h->params.p, (size_t)5 * N * 8, E, h->stream);
        if (e == cudaSuccess && automaton) e = replicate(fire[0], h->fire[h->fire_cur].p, ncell, E, h->stream);
        if (e == cudaSuccess && quad) e = cudaMemsetAsync((void *)lg.planes_q, 0, q_bytes, h->stream);
    }
    if (e == cudaSuccess) e = launch_thresholds(d_x0, N, xyT, h->stream, E), what = "launch_thresholds";
    h->launches += 1;
    if (!app && d_stamp && e == cudaSuccess) e = cudaMemsetAsync(d_stamp, 0, (size_t)E * ncell * 4, h->stream);
    if (app && e == cudaSuccess) {
        what = "append setup";
        e = cudaMemsetAsync(overflow, 0, sizeof(int), h->stream);
        if (e == cudaSuccess && d_stamp) e = cudaMemsetAsync(d_stamp, 0, (size_t)E * ncell * 4, h->stream);
        if (e == cudaSuccess && lg.planes_q && !ens) e = cudaMemsetAsync((void *)lg.planes_q, 0, q_bytes, h->stream);
    }
    int rc = COV_OK;
    for (int64_t t = 1; t <= T && e == cudaSuccess && rc == COV_OK; ++t) {
        const double *cur = t == 1 ? d_x0 : d_Xo + (size_t)(t - 2) * E * n;
        double *next = d_Xo + (size_t)(t - 1) * E * n;
        long long *row = d_st + cols * E * (t - 1);
        if (step_ms && (e = cudaEventRecord(ev[(size_t)t - 1], h->stream)) != cudaSuccess) break;
        if (app && app->offsets && list_of) { // update_POI, each scenario its schedule's rows of this timestep
            int64_t longest = 0;
            for (int64_t q = 0; q < E; ++q) {
                const int64_t *o = app->offsets + list_of[q] * T + (t - 1);
                longest = std::max(longest, o[1] - o[0]);
            }
            what = "append";
            if (longest > 0) {
                if ((e = launch_add_points(mult, cls, d_cell, d_cls, longest, overflow, h->stream, E, d_off + (t - 1),
                                           T, d_list, (long long)ncell)) != cudaSuccess)
                    break;
                h->launches += 1;
            }
        } else if (app && app->offsets) { // update_POI: this timestep's rows of the fire list
            const int64_t q0 = app->offsets[t - 1], q1 = app->offsets[t];
            what = "append";
            if (q1 > q0) {
                if ((e = launch_add_points(mult, cls, d_cell + q0, d_cls + q0, q1 - q0, overflow, h->stream)) != cudaSuccess) break;
                h->launches += 1;
            }
        } else if (app) { // the automaton, its pushes counted into the stats rows (column 4 of each scenario)
            what = "fire step";
            e = E == 1 ? cudaMemsetAsync(row + 4, 0, sizeof(long long), h->stream)
                       : cudaMemset2DAsync(row + 4, (size_t)cols * 8, 0, sizeof(long long), (size_t)E, h->stream);
            if (e != cudaSuccess) break;
            for (int64_t k = 0; k < app->fire_steps[t - 1] && e == cudaSuccess; ++k, ++step) {
                e = launch_fire_step(fire[fire_cur], fire[fire_cur ^ 1], mult, cls, h->g.nx, h->g.ny, app->fire_seed,
                                     (unsigned int)step, d_fp, 1, (unsigned long long *)(row + 4), overflow, h->stream,
                                     E, app->fire_seed_stride, cols);
                if (e == cudaSuccess) fire_cur ^= 1;
                h->launches += 1;
            }
            if (e != cudaSuccess) break;
        }
        what = "rmvCoveredPOI";
        if ((e = launch_remove_covered(mult, cls, lg, xyT, N, (unsigned long long *)(row + 3), h->stream, d_stamp,
                                       (int)t, E, cols)) != cudaSuccess)
            break;
        what = "repack";
        if (!list && (e = launch_pack_planes(mult, cls, lg, (uint32_t *)lg.planes, h->stream, E)) != cudaSuccess) break;
        if (!list && lg.planes_q && (e = launch_requad_plane(lg, (uint32_t *)lg.planes_q, h->stream)) != cudaSuccess)
            break;
        walk.t = t;
        hs.t = t;
        what = "horizon_start";
        if ((e = launch_horizon_start(hs, cur, params, (double *)a.X0, (double *)a.a0, (int *)a.b0, h->stream)) !=
            cudaSuccess)
            break;
        a.seed = seed + (uint64_t)(t - 1) * (uint64_t)S;
        unsigned long long *counter = nullptr;
        if ((rc = take_counter(h, &counter)) != COV_OK) break;
        what = "MADS kernel";
        // one scenario: mads_kernel, its planes staged in shared memory once per CTA
        e = list     ? launch_list_mads(lg, o, cfg, a, S, hs.seed_stride, walk, counter, h->stream)
            : E == 1 ? launch_mads(lg, o, cfg, a, counter, h->stream)
                     : launch_scenario_mads(lg, o, cfg, a, S, hs.seed_stride, counter, h->stream);
        if (e != cudaSuccess) break;
        what = "horizon_commit";
        if ((e = launch_horizon_commit(S, N, a.X_out, a.obj_out, a.stats, next, row, xyT, h->stream, E, cols)) !=
            cudaSuccess)
            break;
        what = "coverage kernel";
        if (list) {
            if ((e = launch_list_eval(lg, o, walk, next, E, d_oo + (t - 1) * E, h->stream)) != cudaSuccess) break;
        } else if (E == 1) {
            if ((rc = take_counter(h, &counter)) != COV_OK) break;
            EvalOut out{};
            out.obj = d_oo + (t - 1);
            LaunchInfo li{};
            if ((e = launch_eval(lg, o, cfg, next, 1, out, counter, h->stream, &li)) != cudaSuccess) break;
        } else if ((e = launch_scenario_eval(lg, o, cfg, next, E, d_oo + (t - 1) * E, h->stream)) != cudaSuccess) {
            break;
        }
        h->launches += list ? 5 : (lg.planes_q ? 7 : 6);
    }
    if (!ens) h->fire_cur = fire_cur; // the automaton steps enqueued stand
    if (e == cudaSuccess && rc == COV_OK && step_ms) e = cudaEventRecord(ev[(size_t)T], h->stream), what = "event";
    if (e == cudaSuccess && rc == COV_OK)
        e = cudaMemcpyAsync(h->h_out, d_Xo, res_bytes, cudaMemcpyDeviceToHost, h->stream), what = "download";
    if (cells_bytes && e == cudaSuccess && rc == COV_OK)
        e = cudaMemcpyAsync((unsigned char *)h->h_out + res_bytes, mult, cells_bytes, cudaMemcpyDeviceToHost, h->stream);
    if (states_bytes && e == cudaSuccess && rc == COV_OK)
        e = cudaMemcpyAsync((unsigned char *)h->h_out + res_bytes + cells_bytes, fire[fire_cur], states_bytes,
                            cudaMemcpyDeviceToHost, h->stream);
    if (app && e == cudaSuccess && rc == COV_OK)
        e = cudaMemcpyAsync(&h->h_small->overflow, overflow, sizeof(int), cudaMemcpyDeviceToHost, h->stream);
    const int n_classes = app ? app->n_classes : h->g.n_classes;
    const double *cw = app ? app->cw : h->g.class_weight;
    if (ens && e == cudaSuccess && rc == COV_OK) e = cudaStreamSynchronize(h->stream), what = "synchronise";
    if (e != cudaSuccess || rc != COV_OK) { // the steps enqueued so far stand: refresh what the host knows of them
        if (rc == COV_OK) rc = fail_cuda(h, e, (std::string(who) + ": " + what).c_str());
        if (ens) { // they only touched the scenarios' copies
            for (cudaEvent_t x : ev) h->ev_pool.push_back(x);
            return rc;
        }
        const std::string msg = h->err;
        if (app) entries_forget(h); // the list's per-timestep history is incomplete
        else entries_note_removals(h);
        // a list-order store: createPOI's order would give other bits, so the store cannot be vouched for any more
        if (rebuild_planes(h, n_classes, cw) != COV_OK || (app && list)) h->have_grid = false;
        for (cudaEvent_t x : ev) h->ev_pool.push_back(x);
        h->err = msg;
        return rc;
    }
    if (!ens) rc = rebuild_planes(h, n_classes, cw); // the one synchronise
    if (rc == COV_OK && app && h->h_small->overflow)
        rc = fail(h, COV_ERR_STATE, std::string(who) + ": internal: an append went past the store's envelope");
    const double *hX = (const double *)h->h_out, *hobj = hX + tn;
    int64_t *hst = (int64_t *)(hobj + T * E);
    const int *hstamp = (const int *)((const unsigned char *)h->h_out + o_stamp);
    if (rc == COV_OK) {
        bool removed = false, pushed = false;
        for (int64_t r = 0; r < T * E; ++r) { // row r: timestep r / E of scenario r % E
            removed |= hst[cols * r + 3] != 0;
            if (app && app->offsets) {
                const int64_t *o = app->offsets + (list_of ? list_of[r % E] * T : 0) + r / E;
                hst[cols * r + 4] = o[1] - o[0];
            }
            if (app) pushed |= hst[cols * r + 4] != 0;
        }
        if (ens) { // the handle's list is untouched
        } else if (automaton && pushed) {
            entries_forget(h); // cov_fire_step: the automaton's order is createPOI's
        } else if (app && app->offsets && h->ent_known) {
            entries_replay(h, *app, T, hstamp);
        } else if (removed) {
            entries_note_removals(h);
        }
        for (int64_t q = 0; q < E; ++q) // timestep-major rows to the scenario-major outputs
            for (int64_t t = 0; t < T; ++t) {
                const size_t src = (size_t)(t * E + q), dst = (size_t)(q * T + t);
                memcpy(X_out + dst * n, hX + src * n, (size_t)n * 8);
                if (obj_out) obj_out[dst] = hobj[src];
                if (stats) memcpy(stats + dst * cols, hst + src * cols, (size_t)cols * 8);
            }
        if (cells_bytes) memcpy(ens->cells_out, (const unsigned char *)h->h_out + res_bytes, cells_bytes);
        if (states_bytes) memcpy(ens->states_out, (const unsigned char *)h->h_out + res_bytes + cells_bytes, states_bytes);
        if (stamps && stamps_out) memcpy(stamps_out, hstamp, (size_t)E * ncell * 4);
        for (int64_t t = 0; step_ms && t < T; ++t) {
            float ms = 0;
            if ((e = cudaEventElapsedTime(&ms, ev[(size_t)t], ev[(size_t)t + 1])) != cudaSuccess) {
                rc = fail_cuda(h, e, (std::string(who) + ": cudaEventElapsedTime").c_str());
                break;
            }
            step_ms[t] = ms;
        }
    }
    for (cudaEvent_t x : ev) h->ev_pool.push_back(x);
    return rc;
}

extern "C" int cov_run_horizon(cov_handle *h, const double *x_start, int64_t T, int64_t S, double spread,
                               int64_t n_iter, double granularity, uint64_t seed, const double *boxes, int64_t n_boxes,
                               double h_focus, double h_max, double *X_out, double *obj_out, int64_t *stats,
                               double *step_ms)
{
    const char *who = "cov_run_horizon";
    if (!h) return fail(nullptr, COV_ERR_INVALID, "NULL handle");
    DeviceGuard dg(h->device);
    OK(check_horizon(h, who, x_start, T, S, spread, n_iter, granularity, boxes, n_boxes, X_out, true));
    if (T == 0) return COV_OK;
    OK(check_mads_limits(h, who, &h->g));
    return run_horizon(h, who, x_start, T, S, spread, n_iter, granularity, seed, boxes, n_boxes, h_focus, h_max, X_out,
                       obj_out, stats, step_ms, nullptr, nullptr, !h->area_exact);
}

extern "C" int cov_run_horizon_ensemble(cov_handle *h, const double *x_starts, int64_t E, int64_t T, int64_t S,
                                        double spread, int64_t n_iter, double granularity, uint64_t seed,
                                        const double *boxes, int64_t n_boxes, double h_focus, double h_max,
                                        double *X_out, double *obj_out, int64_t *stats, double *step_ms,
                                        uint8_t *cells_out)
{
    const char *who = "cov_run_horizon_ensemble";
    if (!h) return fail(nullptr, COV_ERR_INVALID, "NULL handle");
    DeviceGuard dg(h->device);
    OK(check_horizon(h, who, x_starts, T, S, spread, n_iter, granularity, boxes, n_boxes, X_out, true));
    OK(check_ensemble(h, who, E, T, S));
    if (T == 0) return COV_OK;
    OK(check_mads_limits(h, who, &h->g));
    const HorizonEnsemble ens{E, cells_out, nullptr};
    return drop_ensemble(h, run_horizon(h, who, x_starts, T, S, spread, n_iter, granularity, seed, boxes, n_boxes,
                                        h_focus, h_max, X_out, obj_out, stats, step_ms, nullptr, nullptr,
                                        !h->area_exact, &ens));
}

// The cell store's bytes as they are (one download, one synchronise).
static int download_cells(cov_handle *h, std::vector<unsigned char> &m, std::vector<unsigned char> &k,
                          std::vector<unsigned char> *fire_state)
{
    const size_t ncell = (size_t)h->g.nx * h->g.ny;
    m.resize(ncell);
    k.resize(ncell);
    CK(cudaMemcpyAsync(m.data(), h->mult.p, ncell, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(k.data(), h->cls.p, ncell, cudaMemcpyDeviceToHost, h->stream));
    if (fire_state) {
        fire_state->resize(ncell);
        CK(cudaMemcpyAsync(fire_state->data(), h->fire[h->fire_cur].p, ncell, cudaMemcpyDeviceToHost, h->stream));
    }
    CK(cudaStreamSynchronize(h->stream));
    return COV_OK;
}

// cov_run_horizon_points (ens NULL, one schedule, list_of NULL) and cov_run_horizon_points_ensemble (L schedules,
// scenario e on schedule list_of[e]): the checks in cov_run_horizon_points' order, the envelope, the loop.  Every
// scenario starts from the handle's store, so one envelope serves all of them: a cell's bound is the store's
// multiplicity plus the largest count one schedule puts there (a scenario holds only its own schedule).
static int horizon_points(cov_handle *h, const char *who, const double *x_start, int64_t T, int64_t S, double spread,
                          int64_t n_iter, double granularity, uint64_t seed, const double *boxes, int64_t n_boxes,
                          double h_focus, double h_max, const double *pts5, const int64_t *offsets, int64_t L,
                          const int64_t *list_of, double *X_out, double *obj_out, int64_t *stats, double *step_ms,
                          int *last_removed, const HorizonEnsemble *ens)
{
    const int64_t E = ens ? ens->E : 1;
    OK(check_horizon(h, who, x_start, T, S, spread, n_iter, granularity, boxes, n_boxes, X_out, true));
    if (ens) OK(check_ensemble(h, who, E, T, S));
    if (L < 1 || (T > 0 && L > (INT64_MAX - 1) / T))
        return fail(h, COV_ERR_INVALID, std::string(who) + ": L must be >= 1 with L * T + 1 <= 2^63 - 1");
    const int64_t n_off = L * T + 1;
    const std::string bad_offsets = std::string(who) + ": offsets must hold " + (ens ? "L * T + 1" : "T + 1") +
                                    " non-decreasing values from 0";
    if (!offsets || offsets[0] != 0 || T > 0x7fffffffll) return fail(h, COV_ERR_INVALID, bad_offsets);
    for (int64_t q = 1; q < n_off; ++q)
        if (offsets[q] < offsets[q - 1]) return fail(h, COV_ERR_INVALID, bad_offsets);
    const int64_t P = offsets[n_off - 1];
    if (P > 0 && !pts5) return fail(h, COV_ERR_INVALID, std::string(who) + ": pts5 is NULL");
    if (ens && T > 0) {
        if (!list_of) return fail(h, COV_ERR_INVALID, std::string(who) + ": list_of is NULL");
        for (int64_t e = 0; e < E; ++e)
            if (list_of[e] < 0 || list_of[e] >= L)
                return fail(h, COV_ERR_INVALID, std::string(who) + ": list_of must hold E values in [0, L)");
    }
    if (T == 0) return COV_OK;
    HorizonAppend app;
    app.offsets = offsets;
    app.list_of = ens ? list_of : nullptr;
    app.L = L;
    app.n_classes = (h->n_entries == 0 && P > 0) ? 0 : h->g.n_classes; // cov_add_points: an empty store has no weight yet
    for (int k = 0; k < kMaxClasses; ++k) app.cw[k] = h->g.class_weight[k];
    OK(map_points(h, pts5, P, app.cell, app.pcls, app.n_classes, app.cw));
    std::vector<unsigned char> m, k;
    OK(download_cells(h, m, k, nullptr));
    // every cell's multiplicity bound and class: the store's entries plus the most that one schedule puts there
    const size_t ncell = m.size();
    std::vector<int> extra(ncell, 0), cnt(L > 1 ? ncell : 0, 0);
    std::vector<unsigned char> bc(ncell, 0xff);
    for (size_t c = 0; c < ncell; ++c)
        if (m[c]) bc[c] = k[c] & (kMaxClasses - 1);
    int64_t longest = 0;
    for (int64_t l = 0; l < L; ++l) {
        const int64_t q0 = offsets[l * T], q1 = offsets[(l + 1) * T];
        std::vector<int> &mine = L > 1 ? cnt : extra; // one schedule counts straight into the bound
        for (int64_t q = q0; q < q1; ++q) {
            const int c = app.cell[(size_t)q];
            if (bc[c] == 0xff) bc[c] = app.pcls[(size_t)q];
            else if (bc[c] != app.pcls[(size_t)q])
                return fail(h, COV_ERR_INVALID, std::string(who) + ": entries on one cell carry different weights (the "
                                                                   "store's and the schedule's, removals ignored)");
            ++mine[c];
        }
        if (L > 1)
            for (int64_t q = q0; q < q1; ++q) {
                const int c = app.cell[(size_t)q];
                extra[c] = std::max(extra[c], cnt[c]);
                cnt[c] = 0; // the first row on c resets it; the later ones leave zero
            }
        longest = std::max(longest, q1 - q0);
    }
    unsigned max_mult[kMaxClasses] = {0, 0, 0, 0};
    for (size_t c = 0; c < ncell; ++c) {
        const int bound = m[c] + extra[c];
        if (bound > 255)
            return fail(h, COV_ERR_LIMIT, std::string(who) + ": more than 255 list entries on one cell (removals "
                                                             "ignored)");
        if (bound) max_mult[bc[c]] = std::max(max_mult[bc[c]], (unsigned)bound);
    }
    bool list = false;
    OK(horizon_envelope(h, who, app, max_mult, h->n_entries + longest, &list));
    if (ens) { // the scenarios' lists are the caller's to rebuild (last_removed); the handle's stays as it is
        app.stamps = last_removed != nullptr;
        return run_horizon(h, who, x_start, T, S, spread, n_iter, granularity, seed, boxes, n_boxes, h_focus, h_max,
                           X_out, obj_out, stats, step_ms, &app, last_removed, list, ens);
    }
    // the ordered list: removals pending from earlier calls first, and push! appends after the entries already in
    // the list, whatever setter built it (cov_add_points)
    entries_apply_removals(h, m.data());
    if (!h->ent_known && P > 0) {
        entries_from_cells(h, m.data(), k.data());
        h->ent_known = true;
        h->ent_dev_valid = false;
    }
    app.stamps = h->ent_known || last_removed;
    return run_horizon(h, who, x_start, T, S, spread, n_iter, granularity, seed, boxes, n_boxes, h_focus, h_max, X_out,
                       obj_out, stats, step_ms, &app, last_removed, list);
}

extern "C" int cov_run_horizon_points(cov_handle *h, const double *x_start, int64_t T, int64_t S, double spread,
                                      int64_t n_iter, double granularity, uint64_t seed, const double *boxes,
                                      int64_t n_boxes, double h_focus, double h_max, const double *pts5,
                                      const int64_t *offsets, double *X_out, double *obj_out, int64_t *stats,
                                      double *step_ms, int *last_removed)
{
    if (!h) return fail(nullptr, COV_ERR_INVALID, "NULL handle");
    DeviceGuard dg(h->device);
    return horizon_points(h, "cov_run_horizon_points", x_start, T, S, spread, n_iter, granularity, seed, boxes,
                          n_boxes, h_focus, h_max, pts5, offsets, 1, nullptr, X_out, obj_out, stats, step_ms,
                          last_removed, nullptr);
}

extern "C" int cov_run_horizon_points_ensemble(cov_handle *h, const double *x_starts, int64_t E, int64_t T, int64_t S,
                                               double spread, int64_t n_iter, double granularity, uint64_t seed,
                                               const double *boxes, int64_t n_boxes, double h_focus, double h_max,
                                               const double *pts5, const int64_t *offsets, int64_t L,
                                               const int64_t *list_of, double *X_out, double *obj_out, int64_t *stats,
                                               double *step_ms, uint8_t *cells_out, int *last_removed)
{
    if (!h) return fail(nullptr, COV_ERR_INVALID, "NULL handle");
    DeviceGuard dg(h->device);
    const HorizonEnsemble ens{E, cells_out, nullptr};
    return drop_ensemble(h, horizon_points(h, "cov_run_horizon_points_ensemble", x_starts, T, S, spread, n_iter,
                                           granularity, seed, boxes, n_boxes, h_focus, h_max, pts5, offsets, L,
                                           list_of, X_out, obj_out, stats, step_ms, last_removed, &ens));
}

// cov_run_horizon_fire (ens NULL, winds one triple) and cov_run_horizon_fire_ensemble (winds: E triples wind_speed,
// wind_direction, prob_spread): the checks in cov_run_horizon_fire's order, the envelope, the loop.  Every scenario
// starts from the handle's store and automaton state, so one envelope serves all of them.
static int horizon_fire(cov_handle *h, const char *who, const double *x_start, int64_t T, int64_t S, double spread,
                        int64_t n_iter, double granularity, uint64_t seed, const double *boxes, int64_t n_boxes,
                        double h_focus, double h_max, const int64_t *fire_steps, const double *winds,
                        uint64_t fire_seed, uint64_t fire_seed_stride, int64_t first_step, double *X_out,
                        double *obj_out, int64_t *stats, double *step_ms, const HorizonEnsemble *ens)
{
    const int64_t E = ens ? ens->E : 1;
    // after an automaton push the list order is createPOI's, another replay: list-order stores stay refused
    OK(check_horizon(h, who, x_start, T, S, spread, n_iter, granularity, boxes, n_boxes, X_out, false));
    if (ens) OK(check_ensemble(h, who, E, T, S));
    OK(check_fire_store(h, who));
    if (T > 0 && !fire_steps) return fail(h, COV_ERR_INVALID, std::string(who) + ": fire_steps is NULL");
    if (T > 0 && !winds) return fail(h, COV_ERR_INVALID, std::string(who) + ": winds is NULL");
    constexpr int64_t kSteps = 0x100000000ll; // step numbers are 32-bit (cov_fire_step)
    int64_t total = 0;
    for (int64_t t = 0; t < T; ++t) {
        if (fire_steps[t] < 0 || fire_steps[t] > kSteps - total)
            return fail(h, COV_ERR_INVALID, std::string(who) + ": fire_steps must be >= 0 with step numbers below 2^32");
        total += fire_steps[t];
    }
    if (first_step < 0 || first_step > kSteps - total)
        return fail(h, COV_ERR_INVALID, std::string(who) + ": the steps first_step .. first_step + sum(fire_steps) - 1 "
                                                           "must lie in 0 .. 2^32 - 1");
    if (T == 0) return COV_OK;
    std::vector<unsigned char> m, k, st;
    OK(download_cells(h, m, k, &st));
    // a TREE cell ignites at most once and pushes at most one entry per burning Moore neighbour (fire_step_kernel)
    const int nx = h->g.nx, ny = h->g.ny;
    unsigned max_mult[kMaxClasses] = {0, 0, 0, 0};
    int64_t trees = 0;
    for (int j = 1; j <= ny; ++j)
        for (int i = 1; i <= nx; ++i) {
            const size_t c = (size_t)(i - 1) + (size_t)nx * (j - 1);
            const bool tree = total > 0 && st[c] == 1 && i >= 2 && i <= nx - 1 && j >= 2 && j <= ny - 1;
            const unsigned b = m[c] + (tree ? 8u : 0u);
            trees += tree ? 1 : 0;
            if (b > 255)
                return fail(h, COV_ERR_LIMIT, std::string(who) + ": more than 255 list entries on one cell (removals "
                                                                 "ignored)");
            max_mult[0] = std::max(max_mult[0], b);
        }
    HorizonAppend app;
    app.n_classes = 1;
    app.cw[0] = h->g.class_weight[0];
    OK(horizon_envelope(h, who, app, max_mult, h->n_entries + 8 * trees, nullptr));
    std::vector<double> fp((size_t)E * 9);
    for (int64_t e = 0; e < E; ++e) fire_probs(winds[3 * e], winds[3 * e + 1], winds[3 * e + 2], fp.data() + 9 * e);
    app.fire_steps = fire_steps;
    app.fire_p = fp.data();
    app.fire_seed = fire_seed;
    app.fire_seed_stride = fire_seed_stride;
    app.first_step = first_step;
    return run_horizon(h, who, x_start, T, S, spread, n_iter, granularity, seed, boxes, n_boxes, h_focus, h_max, X_out,
                       obj_out, stats, step_ms, &app, nullptr, false, ens);
}

extern "C" int cov_run_horizon_fire(cov_handle *h, const double *x_start, int64_t T, int64_t S, double spread,
                                    int64_t n_iter, double granularity, uint64_t seed, const double *boxes,
                                    int64_t n_boxes, double h_focus, double h_max, const int64_t *fire_steps,
                                    double wind_speed, double wind_direction, double prob_spread, uint64_t fire_seed,
                                    int64_t first_step, double *X_out, double *obj_out, int64_t *stats,
                                    double *step_ms)
{
    if (!h) return fail(nullptr, COV_ERR_INVALID, "NULL handle");
    DeviceGuard dg(h->device);
    const double wind[3] = {wind_speed, wind_direction, prob_spread};
    return horizon_fire(h, "cov_run_horizon_fire", x_start, T, S, spread, n_iter, granularity, seed, boxes, n_boxes,
                        h_focus, h_max, fire_steps, wind, fire_seed, 0, first_step, X_out, obj_out, stats, step_ms,
                        nullptr);
}

extern "C" int cov_run_horizon_fire_ensemble(cov_handle *h, const double *x_starts, int64_t E, int64_t T, int64_t S,
                                             double spread, int64_t n_iter, double granularity, uint64_t seed,
                                             const double *boxes, int64_t n_boxes, double h_focus, double h_max,
                                             const int64_t *fire_steps, const double *winds, uint64_t fire_seed,
                                             uint64_t fire_seed_stride, int64_t first_step, double *X_out,
                                             double *obj_out, int64_t *stats, double *step_ms, uint8_t *cells_out,
                                             uint8_t *states_out)
{
    if (!h) return fail(nullptr, COV_ERR_INVALID, "NULL handle");
    DeviceGuard dg(h->device);
    const HorizonEnsemble ens{E, cells_out, states_out};
    return drop_ensemble(h, horizon_fire(h, "cov_run_horizon_fire_ensemble", x_starts, T, S, spread, n_iter,
                                         granularity, seed, boxes, n_boxes, h_focus, h_max, fire_steps, winds,
                                         fire_seed, fire_seed_stride, first_step, X_out, obj_out, stats, step_ms,
                                         &ens));
}

extern "C" int cov_argmin(cov_handle *h, const double *X, int64_t B, int32_t barrier, double *best_obj,
                          int64_t *best_idx)
{
    if (!h) return fail(nullptr, COV_ERR_INVALID, "NULL handle");
    DeviceGuard dg(h->device);
    OK(check_ready(h, "cov_argmin"));
    if (B < 0 || (B > 0 && !X) || !best_obj || !best_idx) return fail(h, COV_ERR_INVALID, "cov_argmin: bad arguments");
    Winner w;
    const int N = h->o.N;
    const size_t row_bytes = (size_t)3 * N * 8;
    if ((size_t)B * row_bytes > (4u << 20)) { // big sets: the sliced pipeline (H2D of slice k+1 beside the kernel of slice k)
        OK(eval_host(h, X, B, nullptr, nullptr, nullptr, nullptr, nullptr, &w, barrier));
    } else {
        recycle_spans(h);
        const int64_t window = window_rows(B, row_bytes, 1ull << 30);
        OK(ensure(h, h->dX, (size_t)window * row_bytes));
        OK(ensure(h, h->d_obj, (size_t)window * 8));
        OK(ensure(h, h->d_feas, (size_t)window));
        for (int64_t w0 = 0; w0 < B; w0 += window) {
            const int64_t wn = std::min(window, B - w0);
            CK(cudaMemcpyAsync(h->dX.p, X + (size_t)w0 * 3 * N, (size_t)wn * row_bytes, cudaMemcpyHostToDevice, h->stream));
            EvalOut out{};
            out.obj = (double *)h->d_obj.p;
            out.feasible = (unsigned char *)h->d_feas.p;
            OK(launch_on_main(h, (const double *)h->dX.p, wn, out, true));
            OK(enqueue_winner(h, out.obj, out.feasible, wn, barrier));
            CK(cudaStreamSynchronize(h->stream));
            w.offer(h->h_small->win_obj, h->h_small->win_idx, w0);
        }
    }
    *best_obj = w.obj;
    *best_idx = w.idx;
    return COV_OK;
}


// ------------------------------------------------------------------------------------------
// continuous variant: exact union area of the discs (no grid involved)
// ------------------------------------------------------------------------------------------
extern "C" int cov_union_area_batch(cov_handle *h, const double *X, int64_t B, int64_t N, double *area)
{
    if (!h) return fail(nullptr, COV_ERR_INVALID, "NULL handle");
    DeviceGuard dg(h->device);
    if (N < 1 || N > kMaxUavs) return fail(h, COV_ERR_LIMIT, "cov_union_area_batch: N must be 1..1024");
    if (B < 0 || (B > 0 && (!X || !area))) return fail(h, COV_ERR_INVALID, "cov_union_area_batch: bad arguments");
    const size_t row_bytes = (size_t)3 * N * 8;
    const int64_t window = window_rows(B, row_bytes, 256ull << 20);
    OK(ensure(h, h->dX, (size_t)window * row_bytes));
    OK(ensure(h, h->d_obj, (size_t)window * 8));
    for (int64_t w0 = 0; w0 < B; w0 += window) {
        const int64_t wn = std::min(window, B - w0);
        CK(cudaMemcpyAsync(h->dX.p, X + (size_t)w0 * 3 * N, (size_t)wn * row_bytes, cudaMemcpyHostToDevice, h->stream));
        CK(launch_union_area((const double *)h->dX.p, (long long)wn, (int)N, (double *)h->d_obj.p, h->stream));
        h->launches += 1;
        CK(cudaMemcpyAsync(area + w0, h->d_obj.p, (size_t)wn * 8, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
    }
    return COV_OK;
}

// ------------------------------------------------------------------------------------------
// grid-free static objective: the region (domain and covered discs), its batch evaluation and device MADS
// ------------------------------------------------------------------------------------------
extern "C" int cov_set_region(cov_handle *h, double x_lo, double y_lo, double x_hi, double y_hi,
                              const double *covered_xyR, int64_t M)
{
    if (!h) return fail(nullptr, COV_ERR_INVALID, "NULL handle");
    DeviceGuard dg(h->device);
    if (!(std::isfinite(x_lo) && std::isfinite(y_lo) && std::isfinite(x_hi) && std::isfinite(y_hi)) || !(x_hi > x_lo) ||
        !(y_hi > y_lo))
        return fail(h, COV_ERR_INVALID, "cov_set_region: the domain needs finite bounds with x_lo < x_hi, y_lo < y_hi");
    if (M < 0 || (M > 0 && !covered_xyR)) return fail(h, COV_ERR_INVALID, "cov_set_region: bad covered discs");
    if (M > kRegionMaxCovered)
        return fail(h, COV_ERR_LIMIT, "cov_set_region: M = " + std::to_string(M) + " covered discs exceed the " +
                                          std::to_string(kRegionMaxCovered) + " of the kernels' shared-memory plan");
    std::vector<double> x, y, r; // discs of radius <= 0 cover nothing: dropped
    for (int64_t m = 0; m < M; ++m) {
        const double cx = covered_xyR[m], cy = covered_xyR[M + m], R = covered_xyR[2 * M + m];
        if (!(std::isfinite(cx) && std::isfinite(cy) && std::isfinite(R)))
            return fail(h, COV_ERR_INVALID, "cov_set_region: covered disc " + std::to_string(m) + " is not finite");
        if (R > 0) {
            x.push_back(cx);
            y.push_back(cy);
            r.push_back(R);
        }
    }
    const int Mk = (int)r.size();
    std::vector<double> discs(x);
    discs.insert(discs.end(), y.begin(), y.end());
    discs.insert(discs.end(), r.begin(), r.end());
    // built in fresh buffers, swapped in on success: a failing call leaves the earlier region in place
    DevBuf dd, da;
    auto release = [&] {
        if (dd.p) cudaFree(dd.p);
        if (da.p) cudaFree(da.p);
    };
    int rc = ensure(h, dd, discs.size() * 8);
    if (rc == COV_OK) rc = ensure(h, da, (size_t)kRegionMaxArcs * sizeof(RegionArc));
    if (rc == COV_OK) rc = ensure(h, h->region_count, sizeof(int));
    if (rc != COV_OK) {
        release();
        return rc;
    }
    RegionDesc rd{x_lo, y_lo, x_hi, y_hi, Mk, 0, (const double *)dd.p, (const RegionArc *)da.p};
    int K = 0;
    cudaError_t e = cudaSuccess;
    if (Mk > 0) e = cudaMemcpyAsync(dd.p, discs.data(), discs.size() * 8, cudaMemcpyHostToDevice, h->stream);
    if (e == cudaSuccess && Mk > 0) e = launch_region_arcs(rd, (RegionArc *)da.p, kRegionMaxArcs, (int *)h->region_count.p, h->stream);
    if (e == cudaSuccess && Mk > 0) {
        h->launches += 1;
        e = cudaMemcpyAsync(&h->h_small->region_arcs, h->region_count.p, sizeof(int), cudaMemcpyDeviceToHost, h->stream);
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
    if (e != cudaSuccess) {
        release();
        return fail_cuda(h, e, "cov_set_region");
    }
    if (Mk > 0) K = h->h_small->region_arcs;
    if (K > kRegionMaxArcs) {
        release();
        return fail(h, COV_ERR_LIMIT, "cov_set_region: the covered discs' boundary has " + std::to_string(K) +
                                          " arcs inside the domain, more than the " + std::to_string(kRegionMaxArcs) +
                                          " of the kernels' shared-memory plan");
    }
    std::swap(h->region_discs, dd);
    std::swap(h->region_arcs, da);
    release(); // the earlier region's buffers
    rd.K = K;
    h->region = rd;
    h->have_region = true;
    return COV_OK;
}

static int check_region(cov_handle *h, const char *who)
{
    if (!h->have_region) return fail(h, COV_ERR_STATE, std::string(who) + ": no region set");
    if (!h->have_params) return fail(h, COV_ERR_STATE, std::string(who) + ": no parameters set");
    if (h->o.N > kRegionMaxUavs)
        return fail(h, COV_ERR_LIMIT, std::string(who) + ": N = " + std::to_string(h->o.N) + " exceeds the " +
                                          std::to_string(kRegionMaxUavs) + " discs of a candidate the kernels take");
    return COV_OK;
}

extern "C" int cov_eval_region_batch(cov_handle *h, const double *X, int64_t B, double *obj, double *area,
                                     uint8_t *feasible, int32_t barrier, double *best_obj, int64_t *best_idx)
{
    if (!h) return fail(nullptr, COV_ERR_INVALID, "NULL handle");
    DeviceGuard dg(h->device);
    OK(check_region(h, "cov_eval_region_batch"));
    if (B < 0 || (B > 0 && !X) || (!best_obj != !best_idx))
        return fail(h, COV_ERR_INVALID, "cov_eval_region_batch: bad arguments");
    const bool want_best = best_obj != nullptr;
    const int N = h->o.N;
    const size_t row_bytes = (size_t)3 * N * 8;
    const int64_t window = window_rows(B, row_bytes, 1ull << 30);
    OK(ensure(h, h->dX, (size_t)window * row_bytes));
    OK(ensure(h, h->d_obj, (size_t)window * 8));
    OK(ensure(h, h->d_area, (size_t)window * 8));
    OK(ensure(h, h->d_feas, (size_t)window));
    Winner w;
    recycle_spans(h);
    for (int64_t w0 = 0; w0 < B; w0 += window) {
        const int64_t wn = std::min(window, B - w0);
        CK(cudaMemcpyAsync(h->dX.p, X + (size_t)w0 * 3 * N, (size_t)wn * row_bytes, cudaMemcpyHostToDevice, h->stream));
        double *d_obj = (double *)h->d_obj.p, *d_area = (double *)h->d_area.p;
        unsigned char *d_feas = (unsigned char *)h->d_feas.p;
        OK(timed_launch(h, true, nullptr, "cov_eval_region_batch: kernel launch",
                        "cov_eval_region_batch: the region does not fit the shared-memory plan", [&] {
                            return launch_region_eval(h->region, h->o, h->cfg, (const double *)h->dX.p, wn, d_obj,
                                                      area ? d_area : nullptr, d_feas, h->stream);
                        }));
        if (want_best) OK(enqueue_winner(h, d_obj, d_feas, wn, barrier));
        if (obj) CK(cudaMemcpyAsync(obj + w0, d_obj, (size_t)wn * 8, cudaMemcpyDeviceToHost, h->stream));
        if (area) CK(cudaMemcpyAsync(area + w0, d_area, (size_t)wn * 8, cudaMemcpyDeviceToHost, h->stream));
        if (feasible) CK(cudaMemcpyAsync(feasible + w0, d_feas, (size_t)wn, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        if (want_best) w.offer(h->h_small->win_obj, h->h_small->win_idx, w0);
    }
    if (want_best) {
        *best_obj = w.obj;
        *best_idx = w.idx;
    }
    return COV_OK;
}

extern "C" int cov_mads_solve_batch_region(cov_handle *h, const double *X0, int64_t S, int64_t n_iter,
                                           double granularity, uint64_t seed, double *X_out, double *obj_out,
                                           int64_t *stats)
{
    if (!h) return fail(nullptr, COV_ERR_INVALID, "NULL handle");
    DeviceGuard dg(h->device);
    OK(check_region(h, "cov_mads_solve_batch_region"));
    return mads_solve_batch(h, true, X0, S, n_iter, granularity, seed, X_out, obj_out, stats);
}

// cov_run_horizon's loop on the region objective (DESIGN.md 18), all enqueued before one synchronise.  Per timestep
// five launches: the covered set's step (launch_cover_arcs), horizon_start_kernel, the S solves (launch_cover_mads),
// horizon_commit_kernel (its thresholds go to scratch: nothing reads them) and the objective of the winner
// (launch_cover_eval).  The covered set grows in a buffer of the call; the handle gets it only when every timestep
// passed, and otherwise its parameters are copied back from the snapshot taken when the call started.
extern "C" int cov_run_horizon_region(cov_handle *h, const double *x_start, int64_t T, int64_t S, double spread,
                                      int64_t n_iter, double granularity, uint64_t seed, const double *boxes,
                                      int64_t n_boxes, double h_focus, double h_max, double *X_out, double *obj_out,
                                      int64_t *stats, double *step_ms)
{
    const char *who = "cov_run_horizon_region";
    if (!h) return fail(nullptr, COV_ERR_INVALID, "NULL handle");
    DeviceGuard dg(h->device);
    OK(check_region(h, who));
    if (!h->o.use_cons3)
        return fail(h, COV_ERR_STATE, std::string(who) + ": the parameters have no previous swarm (cons3 is off)");
    OK(check_mads_limits(h, who, nullptr));
    const int N = h->o.N, n = 3 * N, M0 = h->region.M;
    if (T > 0 && T > (kRegionMaxCovered - M0) / N) // discs with R <= 0 count: how many go is known on the device only
        return fail(h, COV_ERR_LIMIT, std::string(who) + ": M0 + T N = " + std::to_string(M0) + " + " +
                                          std::to_string(T) + " x " + std::to_string(N) + " covered discs exceed the " +
                                          std::to_string(kRegionMaxCovered) + " of the kernels' shared-memory plan");
    OK(check_horizon_args(h, who, x_start, T, S, spread, n_iter, granularity, boxes, n_boxes, X_out));
    if (T == 0) return COV_OK;
    for (int q = 0; q < n; ++q)
        if (!std::isfinite(x_start[q])) return fail(h, COV_ERR_INVALID, std::string(who) + ": x_start is not finite");
    const int pitch = M0 + (int)T * N;
    // in: [pow10 | x_start: n | boxes: 4 n_boxes | ctl: 4 ints | the solves' inputs]; out: [the solves' outputs |
    // X_out: T n | obj_out: T | stats: T x 4 | the parameters at the call: 5N | thresholds: n | covered discs: 3 pitch]
    const size_t tn = (size_t)T * n, o_x = kPow10Bytes, o_box = o_x + (size_t)n * 8;
    const size_t o_ctl = o_box + (size_t)n_boxes * 32, o_X0 = o_ctl + 16;
    const size_t o_par = tn * 8 + (size_t)T * 8 + (size_t)T * 32, o_xyT = o_par + (size_t)5 * N * 8;
    const size_t o_disc = o_xyT + (size_t)n * 8, dev_bytes = o_disc + (size_t)3 * pitch * 8;
    std::vector<unsigned char> hin(o_X0);
    MadsArgs a;
    OK(mads_buffers(h, o_X0, S, n, dev_bytes, hin, a));
    memcpy(hin.data() + o_x, x_start, (size_t)n * 8);
    if (n_boxes) memcpy(hin.data() + o_box, boxes, (size_t)n_boxes * 32);
    const int ctl0[4] = {M0, h->region.K, 0, 0};
    memcpy(hin.data() + o_ctl, ctl0, sizeof(ctl0));
    OK(ensure_pinned(h, &h->h_out, &h->h_out_cap, o_par + sizeof(ctl0)));
    DevBuf dd, da; // the region's discs and arcs after the call, swapped in on success as cov_set_region does
    auto release = [&] {
        if (dd.p) cudaFree(dd.p);
        if (da.p) cudaFree(da.p);
    };
    int rc = ensure(h, dd, (size_t)3 * pitch * 8);
    if (rc == COV_OK) rc = ensure(h, da, (size_t)kRegionMaxArcs * sizeof(RegionArc));
    if (rc != COV_OK) {
        release();
        return rc;
    }
    unsigned char *din = (unsigned char *)h->mads_in.p;
    const double *d_x0 = (const double *)(din + o_x);
    double *d_Xo = (double *)(a.stats + 4 * S), *d_oo = d_Xo + tn;
    long long *d_st = (long long *)(d_oo + T);
    unsigned char *dres = (unsigned char *)d_Xo;
    double *params = (double *)h->params.p, *backup = (double *)(dres + o_par), *xyT = (double *)(dres + o_xyT);
    const RegionDesc &r = h->region;
    const CoverSet cs{r.x_lo, r.y_lo, r.x_hi, r.y_hi, (double *)(dres + o_disc), (RegionArc *)da.p, pitch,
                      (int *)(din + o_ctl)};
    a.n_iter = n_iter;
    a.granularity = granularity;
    a.ordered = 0;
    HorizonStep hs{};
    hs.N = N;
    hs.n_boxes = (int)n_boxes;
    hs.S = S;
    hs.E = 1;
    hs.spread = spread;
    hs.granularity = granularity;
    hs.seed = seed;
    hs.pow10 = a.pow10;
    hs.boxes = (const double *)(din + o_box);
    hs.h_focus = h_focus;
    hs.h_max = h_max;
    hs.tan_half_fov = h->o.tan_half_fov;
    std::vector<cudaEvent_t> ev;
    if (step_ms)
        for (int64_t t = 0; t <= T; ++t) ev.push_back(get_event(h));

    cudaError_t e = cudaMemcpyAsync(din, hin.data(), o_X0, cudaMemcpyHostToDevice, h->stream);
    const char *what = "upload";
    bool saved = false; // the parameters' snapshot is enqueued
    if (e == cudaSuccess) {
        what = "parameters";
        e = cudaMemcpyAsync(backup, params, (size_t)5 * N * 8, cudaMemcpyDeviceToDevice, h->stream);
        saved = e == cudaSuccess;
    }
    if (e == cudaSuccess && M0 > 0) // the handle's discs at the call's pitch
        e = cudaMemcpy2DAsync(cs.discs, (size_t)pitch * 8, r.discs, (size_t)M0 * 8, (size_t)M0 * 8, 3,
                              cudaMemcpyDeviceToDevice, h->stream), what = "covered discs";
    for (int64_t t = 1; t <= T && e == cudaSuccess && rc == COV_OK; ++t) {
        const double *cur = t == 1 ? d_x0 : d_Xo + (size_t)(t - 2) * n;
        double *next = d_Xo + (size_t)(t - 1) * n;
        long long *row = d_st + 4 * (t - 1);
        if (step_ms && (e = cudaEventRecord(ev[(size_t)t - 1], h->stream)) != cudaSuccess) break;
        what = "covered set";
        if ((e = launch_cover_arcs(cs, cur, N, t, row, h->stream)) != cudaSuccess) break;
        hs.t = t;
        what = "horizon_start";
        if ((e = launch_horizon_start(hs, cur, params, (double *)a.X0, (double *)a.a0, (int *)a.b0, h->stream)) !=
            cudaSuccess)
            break;
        a.seed = seed + (uint64_t)(t - 1) * (uint64_t)S;
        unsigned long long *counter = nullptr;
        if ((rc = take_counter(h, &counter)) != COV_OK) break;
        what = "MADS kernel";
        if ((e = launch_cover_mads(cs, h->o, h->cfg, a, counter, h->stream)) != cudaSuccess) break;
        what = "horizon_commit";
        if ((e = launch_horizon_commit(S, N, a.X_out, a.obj_out, a.stats, next, row, xyT, h->stream)) != cudaSuccess)
            break;
        what = "objective";
        if ((e = launch_cover_eval(cs, h->o, next, d_oo + (t - 1), h->stream)) != cudaSuccess) break;
        h->launches += 5;
    }
    if (e == cudaSuccess && rc == COV_OK && step_ms) e = cudaEventRecord(ev[(size_t)T], h->stream), what = "event";
    unsigned char *hres = (unsigned char *)h->h_out;
    if (e == cudaSuccess && rc == COV_OK)
        e = cudaMemcpyAsync(hres, d_Xo, o_par, cudaMemcpyDeviceToHost, h->stream), what = "download";
    if (e == cudaSuccess && rc == COV_OK)
        e = cudaMemcpyAsync(hres + o_par, cs.ctl, sizeof(ctl0), cudaMemcpyDeviceToHost, h->stream);
    if (e == cudaSuccess && rc == COV_OK) e = cudaStreamSynchronize(h->stream), what = "synchronise";
    const int *ctl = (const int *)(hres + o_par); // M_T, K_T, failure, its timestep
    if (e == cudaSuccess && rc == COV_OK && ctl[2] == kCoverBadDisc)
        rc = fail(h, COV_ERR_INVALID, std::string(who) + ": timestep " + std::to_string(ctl[3]) +
                                          ": a disc of the swarm is not finite");
    else if (e == cudaSuccess && rc == COV_OK && ctl[2] == kCoverManyArcs)
        rc = fail(h, COV_ERR_LIMIT, std::string(who) + ": timestep " + std::to_string(ctl[3]) +
                                        ": the covered discs' boundary has " + std::to_string(ctl[1]) +
                                        " arcs inside the domain, more than the " + std::to_string(kRegionMaxArcs) +
                                        " of the kernels' shared-memory plan");
    // success: the final discs at their own pitch, cov_set_region's layout
    if (e == cudaSuccess && rc == COV_OK && ctl[0] > 0)
        e = cudaMemcpy2DAsync(dd.p, (size_t)ctl[0] * 8, cs.discs, (size_t)pitch * 8, (size_t)ctl[0] * 8, 3,
                              cudaMemcpyDeviceToDevice, h->stream), what = "covered discs";
    if (e != cudaSuccess || rc != COV_OK) { // the region and the parameters as before the call
        if (rc == COV_OK)
            rc = e == cudaErrorInvalidConfiguration
                     ? fail(h, COV_ERR_LIMIT, std::string(who) + ": one warp of the solver does not fit the shared memory")
                     : fail_cuda(h, e, (std::string(who) + ": " + what).c_str());
        const std::string msg = h->err;
        if (saved) {
            (void)cudaMemcpyAsync(params, backup, (size_t)5 * N * 8, cudaMemcpyDeviceToDevice, h->stream);
            (void)cudaStreamSynchronize(h->stream);
            (void)cudaGetLastError();
        }
        release();
        for (cudaEvent_t x : ev) h->ev_pool.push_back(x);
        h->err = msg;
        return rc;
    }
    std::swap(h->region_discs, dd);
    std::swap(h->region_arcs, da);
    release(); // the earlier region's buffers
    h->region = RegionDesc{r.x_lo, r.y_lo, r.x_hi, r.y_hi, ctl[0], ctl[1], (const double *)h->region_discs.p,
                           (const RegionArc *)h->region_arcs.p};
    const double *hX = (const double *)hres, *hobj = hX + tn;
    const int64_t *hst = (const int64_t *)(hobj + T);
    memcpy(X_out, hX, tn * 8);
    if (obj_out) memcpy(obj_out, hobj, (size_t)T * 8);
    if (stats) memcpy(stats, hst, (size_t)T * 32);
    for (int64_t t = 0; step_ms && t < T && rc == COV_OK; ++t) {
        float ms = 0;
        if ((e = cudaEventElapsedTime(&ms, ev[(size_t)t], ev[(size_t)t + 1])) != cudaSuccess)
            rc = fail_cuda(h, e, (std::string(who) + ": cudaEventElapsedTime").c_str());
        step_ms[t] = ms;
    }
    for (cudaEvent_t x : ev) h->ev_pool.push_back(x);
    return rc;
}

// ------------------------------------------------------------------------------------------
// streams, memory, timing
// ------------------------------------------------------------------------------------------
extern "C" int cov_sync(cov_handle *h)
{
    if (!h) return fail(nullptr, COV_ERR_INVALID, "NULL handle");
    DeviceGuard dg(h->device);
    CK(cudaStreamSynchronize(h->s_in));
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaStreamSynchronize(h->s_out));
    return COV_OK;
}
extern "C" void *cov_stream(cov_handle *h) { return h ? (void *)h->stream : nullptr; }
extern "C" int cov_set_stream(cov_handle *h, void *stream)
{
    if (!h) return fail(nullptr, COV_ERR_INVALID, "NULL handle");
    DeviceGuard dg(h->device);
    CK(cudaStreamSynchronize(h->stream));
    h->stream = stream ? (cudaStream_t)stream : h->own_stream;
    return COV_OK;
}
extern "C" int cov_host_alloc(cov_handle *h, int64_t bytes, void **out)
{
    if (!h || !out || bytes < 0) return fail(h, COV_ERR_INVALID, "cov_host_alloc: bad arguments");
    DeviceGuard dg(h->device);
    *out = nullptr;
    cudaError_t e = cudaMallocHost(out, (size_t)std::max<int64_t>(bytes, 1));
    if (e != cudaSuccess) {
        (void)cudaGetLastError();
        return fail(h, COV_ERR_NOMEM, std::string("cudaMallocHost: ") + cudaGetErrorString(e));
    }
    return COV_OK;
}
extern "C" int cov_host_free(cov_handle *h, void *p)
{
    if (!h) return fail(nullptr, COV_ERR_INVALID, "NULL handle");
    DeviceGuard dg(h->device);
    if (p) CK(cudaFreeHost(p));
    return COV_OK;
}
extern "C" int cov_device_alloc(cov_handle *h, int64_t bytes, void **out)
{
    if (!h || !out || bytes < 0) return fail(h, COV_ERR_INVALID, "cov_device_alloc: bad arguments");
    DeviceGuard dg(h->device);
    *out = nullptr;
    cudaError_t e = cudaMalloc(out, (size_t)std::max<int64_t>(bytes, 1));
    if (e != cudaSuccess) {
        (void)cudaGetLastError();
        return fail(h, COV_ERR_NOMEM, std::string("cudaMalloc: ") + cudaGetErrorString(e));
    }
    return COV_OK;
}
extern "C" int cov_device_free(cov_handle *h, void *p)
{
    if (!h) return fail(nullptr, COV_ERR_INVALID, "NULL handle");
    DeviceGuard dg(h->device);
    if (p) CK(cudaFree(p));
    return COV_OK;
}
extern "C" int cov_memcpy_h2d(cov_handle *h, void *dst, const void *src, int64_t bytes)
{
    if (!h || bytes < 0) return fail(h, COV_ERR_INVALID, "cov_memcpy_h2d: bad arguments");
    DeviceGuard dg(h->device);
    CK(cudaMemcpyAsync(dst, src, (size_t)bytes, cudaMemcpyHostToDevice, h->stream));
    return COV_OK;
}
extern "C" int cov_memcpy_d2h(cov_handle *h, void *dst, const void *src, int64_t bytes)
{
    if (!h || bytes < 0) return fail(h, COV_ERR_INVALID, "cov_memcpy_d2h: bad arguments");
    DeviceGuard dg(h->device);
    CK(cudaMemcpyAsync(dst, src, (size_t)bytes, cudaMemcpyDeviceToHost, h->stream));
    return COV_OK;
}
extern "C" int64_t cov_launch_count(const cov_handle *h) { return h ? h->launches : 0; }

extern "C" int64_t cov_get_trace(const cov_handle *h, double *ms, int64_t cap)
{
    if (!h) return 0;
    const int64_t n = (int64_t)h->trace_ms.size();
    for (int64_t k = 0; k < n && k < cap && ms; ++k) ms[k] = h->trace_ms[k];
    return n;
}

extern "C" int cov_last_kernel_ms(cov_handle *h, double *ms)
{
    if (!h || !ms) return fail(h, COV_ERR_INVALID, "cov_last_kernel_ms: bad arguments");
    DeviceGuard dg(h->device);
    if (h->last_call_ms_cache < 0 || h->kernel_spans.size() > h->last_call_begin) {
        const double before = h->last_call_ms_cache < 0 ? 0 : h->last_call_ms_cache;
        CK(drain_spans(h));
        h->last_call_ms_cache += before;
    }
    *ms = h->last_call_ms_cache;
    return COV_OK;
}

extern "C" int cov_last_launch(const cov_handle *h, cov_launch_info *out)
{
    if (!h || !out) return COV_ERR_INVALID;
    if (h->last_info.block == 0) return COV_ERR_STATE;
    out->kernel = h->last_info.kernel;
    out->grid = h->last_info.grid;
    out->block = h->last_info.block;
    out->smem_bytes = h->last_info.smem_bytes;
    out->band_rows = h->last_info.band_rows;
    out->planes_in_smem = h->last_info.planes_in_smem;
    out->multi = h->last_info.multi;
    out->chunk = h->last_info.chunk;
    out->max_warps = h->last_info.max_warps;
    out->plane_mode = h->last_info.plane_mode;
    return COV_OK;
}

extern "C" int cov_kernel_time_total(cov_handle *h, double *ms, int64_t *launches)
{
    if (!h) return fail(nullptr, COV_ERR_INVALID, "NULL handle");
    DeviceGuard dg(h->device);
    const double keep = h->last_call_ms_cache;
    const bool pending = h->kernel_spans.size() > h->last_call_begin;
    CK(drain_spans(h));
    if (keep >= 0 && pending) h->last_call_ms_cache += keep;
    else if (keep >= 0 && !pending) h->last_call_ms_cache = keep;
    if (ms) *ms = h->drained_ms;
    if (launches) *launches = h->drained_launches;
    return COV_OK;
}

extern "C" int cov_generate_candidates(cov_handle *h, double *dX, int64_t B, int64_t N, uint64_t seed,
                                       int64_t first_index, double lx, double ly, double h_min, double h_max,
                                       double tan_half_fov)
{
    if (!h) return fail(nullptr, COV_ERR_INVALID, "NULL handle");
    DeviceGuard dg(h->device);
    if (B < 0 || N < 1 || N > kMaxUavs || (B > 0 && !dX)) return fail(h, COV_ERR_INVALID, "cov_generate_candidates: bad arguments");
    CK(launch_generate(dX, (long long)B, (int)N, seed, (long long)first_index, lx, ly, h_min, h_max, tan_half_fov,
                       h->stream));
    h->launches += 1;
    return COV_OK;
}

// ------------------------------------------------------------------------------------------
// several GPUs of one box: contiguous candidate slices, one host thread per device
// ------------------------------------------------------------------------------------------
struct cov_multi {
    std::vector<cov_handle *> hs;
    std::string err;
};

extern "C" int cov_multi_create(const int *devices, int n, cov_multi **out)
{
    if (!out || n < 1 || !devices) return fail(nullptr, COV_ERR_INVALID, "cov_multi_create: bad arguments");
    *out = nullptr;
    cov_multi *m = new cov_multi();
    for (int k = 0; k < n; ++k) {
        cov_handle *h = nullptr;
        int rc = cov_create(devices[k], &h);
        if (rc != COV_OK) {
            for (cov_handle *q : m->hs) cov_destroy(q);
            delete m;
            return rc;
        }
        m->hs.push_back(h);
    }
    *out = m;
    return COV_OK;
}
extern "C" void cov_multi_destroy(cov_multi *m)
{
    if (!m) return;
    for (cov_handle *h : m->hs) cov_destroy(h);
    delete m;
}
extern "C" const char *cov_multi_last_error(const cov_multi *m) { return m ? m->err.c_str() : g_err_nohandle.c_str(); }
extern "C" int cov_multi_size(const cov_multi *m) { return m ? (int)m->hs.size() : 0; }
extern "C" cov_handle *cov_multi_handle(cov_multi *m, int k)
{
    return (m && k >= 0 && k < (int)m->hs.size()) ? m->hs[k] : nullptr;
}

static void shard(int64_t B, int G, int k, int64_t &b0, int64_t &bn)
{
    const int64_t per = (B + G - 1) / G; // ceil(B/G), SURVEY.md 8e
    b0 = std::min<int64_t>(B, per * k);
    bn = std::min<int64_t>(B, b0 + per) - b0;
}

// run(k, handle, candidates, b0, bn) on every non-empty shard k of X, one host thread per device; the first shard that
// failed is the call's error.
template <class Run>
static int run_shards(cov_multi *m, const double *X, int64_t B, Run &&run)
{
    const int G = (int)m->hs.size();
    std::vector<int> rcs((size_t)G, COV_OK);
    std::vector<std::thread> th;
    for (int k = 0; k < G; ++k)
        th.emplace_back([&, k]() {
            int64_t b0, bn;
            shard(B, G, k, b0, bn);
            cov_handle *h = m->hs[k];
            if (bn > 0) rcs[k] = run(k, h, X + (size_t)b0 * 3 * (h->have_params ? h->o.N : 0), b0, bn);
        });
    for (auto &t : th) t.join();
    for (int k = 0; k < G; ++k)
        if (rcs[k] != COV_OK) {
            m->err = "device shard " + std::to_string(k) + ": " + m->hs[k]->err;
            return rcs[k];
        }
    return COV_OK;
}

extern "C" int cov_multi_eval_batch(cov_multi *m, const double *X, int64_t B, double *obj, int64_t *count,
                                    uint8_t *feasible)
{
    if (!m) return fail(nullptr, COV_ERR_INVALID, "NULL multi handle");
    if (B < 0 || (B > 0 && (!X || !obj))) {
        m->err = "cov_multi_eval_batch: bad arguments";
        return COV_ERR_INVALID;
    }
    return run_shards(m, X, B, [&](int, cov_handle *h, const double *Xk, int64_t b0, int64_t bn) {
        return cov_eval_batch(h, Xk, bn, obj + b0, count ? count + b0 : nullptr, feasible ? feasible + b0 : nullptr);
    });
}

// Scenarios b0 .. b0 + bn - 1 on shard k with the keys they have in the single-device call.
extern "C" int cov_multi_run_horizon_ensemble(cov_multi *m, const double *x_starts, int64_t E, int64_t T, int64_t S,
                                              double spread, int64_t n_iter, double granularity, uint64_t seed,
                                              const double *boxes, int64_t n_boxes, double h_focus, double h_max,
                                              double *X_out, double *obj_out, int64_t *stats, uint8_t *cells_out)
{
    if (!m) return fail(nullptr, COV_ERR_INVALID, "NULL multi handle");
    if (E < 1 || T < 0 || (T > 0 && (!x_starts || !X_out))) {
        m->err = "cov_multi_run_horizon_ensemble: bad arguments";
        return COV_ERR_INVALID;
    }
    return run_shards(m, x_starts, E, [&](int, cov_handle *h, const double *Xk, int64_t b0, int64_t bn) {
        const size_t n = h->have_params ? 3 * (size_t)h->o.N : 0, ncell = (size_t)h->g.nx * h->g.ny;
        const size_t r0 = (size_t)b0 * (size_t)T;
        return cov_run_horizon_ensemble(h, Xk, bn, T, S, spread, n_iter, granularity,
                                        seed + (uint64_t)b0 * (uint64_t)T * (uint64_t)S, boxes, n_boxes, h_focus, h_max,
                                        X_out + r0 * n, obj_out ? obj_out + r0 : nullptr, stats ? stats + r0 * 4 : nullptr,
                                        nullptr, cells_out ? cells_out + (size_t)b0 * ncell : nullptr);
    });
}

// Scenarios b0 .. b0 + bn - 1 on shard k with the keys, fire seeds and winds they have in the single-device call.
extern "C" int cov_multi_run_horizon_fire_ensemble(cov_multi *m, const double *x_starts, int64_t E, int64_t T, int64_t S,
                                                   double spread, int64_t n_iter, double granularity, uint64_t seed,
                                                   const double *boxes, int64_t n_boxes, double h_focus, double h_max,
                                                   const int64_t *fire_steps, const double *winds, uint64_t fire_seed,
                                                   uint64_t fire_seed_stride, int64_t first_step, double *X_out,
                                                   double *obj_out, int64_t *stats, uint8_t *cells_out,
                                                   uint8_t *states_out)
{
    if (!m) return fail(nullptr, COV_ERR_INVALID, "NULL multi handle");
    if (E < 1 || T < 0 || (T > 0 && (!x_starts || !X_out || !winds))) {
        m->err = "cov_multi_run_horizon_fire_ensemble: bad arguments";
        return COV_ERR_INVALID;
    }
    return run_shards(m, x_starts, E, [&](int, cov_handle *h, const double *Xk, int64_t b0, int64_t bn) {
        const size_t n = h->have_params ? 3 * (size_t)h->o.N : 0, ncell = (size_t)h->g.nx * h->g.ny;
        const size_t r0 = (size_t)b0 * (size_t)T;
        return cov_run_horizon_fire_ensemble(h, Xk, bn, T, S, spread, n_iter, granularity,
                                             seed + (uint64_t)b0 * (uint64_t)T * (uint64_t)S, boxes, n_boxes, h_focus,
                                             h_max, fire_steps, winds ? winds + 3 * b0 : nullptr,
                                             fire_seed + (uint64_t)b0 * fire_seed_stride, fire_seed_stride, first_step,
                                             X_out + r0 * n, obj_out ? obj_out + r0 : nullptr,
                                             stats ? stats + r0 * 5 : nullptr, nullptr,
                                             cells_out ? cells_out + (size_t)b0 * ncell : nullptr,
                                             states_out ? states_out + (size_t)b0 * ncell : nullptr);
    });
}

// Scenarios b0 .. b0 + bn - 1 on shard k with the keys and schedules they have in the single-device call.
extern "C" int cov_multi_run_horizon_points_ensemble(cov_multi *m, const double *x_starts, int64_t E, int64_t T,
                                                     int64_t S, double spread, int64_t n_iter, double granularity,
                                                     uint64_t seed, const double *boxes, int64_t n_boxes,
                                                     double h_focus, double h_max, const double *pts5,
                                                     const int64_t *offsets, int64_t L, const int64_t *list_of,
                                                     double *X_out, double *obj_out, int64_t *stats,
                                                     uint8_t *cells_out, int *last_removed)
{
    if (!m) return fail(nullptr, COV_ERR_INVALID, "NULL multi handle");
    if (E < 1 || T < 0 || (T > 0 && (!x_starts || !X_out || !list_of))) {
        m->err = "cov_multi_run_horizon_points_ensemble: bad arguments";
        return COV_ERR_INVALID;
    }
    return run_shards(m, x_starts, E, [&](int, cov_handle *h, const double *Xk, int64_t b0, int64_t bn) {
        const size_t n = h->have_params ? 3 * (size_t)h->o.N : 0, ncell = (size_t)h->g.nx * h->g.ny;
        const size_t r0 = (size_t)b0 * (size_t)T;
        return cov_run_horizon_points_ensemble(h, Xk, bn, T, S, spread, n_iter, granularity,
                                               seed + (uint64_t)b0 * (uint64_t)T * (uint64_t)S, boxes, n_boxes,
                                               h_focus, h_max, pts5, offsets, L, list_of ? list_of + b0 : nullptr,
                                               X_out + r0 * n, obj_out ? obj_out + r0 : nullptr,
                                               stats ? stats + r0 * 5 : nullptr, nullptr,
                                               cells_out ? cells_out + (size_t)b0 * ncell : nullptr,
                                               last_removed ? last_removed + (size_t)b0 * ncell : nullptr);
    });
}

extern "C" int cov_multi_argmin(cov_multi *m, const double *X, int64_t B, int32_t barrier, double *best_obj,
                                int64_t *best_idx)
{
    if (!m) return fail(nullptr, COV_ERR_INVALID, "NULL multi handle");
    if (B < 0 || (B > 0 && !X) || !best_obj || !best_idx) {
        m->err = "cov_multi_argmin: bad arguments";
        return COV_ERR_INVALID;
    }
    const int G = (int)m->hs.size();
    std::vector<double> bo((size_t)G, INFINITY);
    std::vector<int64_t> bi((size_t)G, -1);
    OK(run_shards(m, X, B, [&](int k, cov_handle *h, const double *Xk, int64_t b0, int64_t bn) {
        const int rc = cov_argmin(h, Xk, bn, barrier, &bo[k], &bi[k]);
        if (rc == COV_OK && bi[k] >= 0) bi[k] += b0;
        return rc;
    }));
    Winner w; // 16-byte (min, index) pair per GPU, host gather
    for (int k = 0; k < G; ++k) w.offer(bo[k], bi[k]);
    *best_obj = w.obj;
    *best_idx = w.idx;
    return COV_OK;
}
