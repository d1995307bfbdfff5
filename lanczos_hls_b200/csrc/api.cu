// api.cu -- the C ABI (include/lanczos_b200.h), plan cache, and the host drivers.
//
// Host driver = what sim_tb does around the two resampler calls in the reference
// (full_TB.h:99-180) minus the PNG codec: move pixels in, run the resampler, move pixels out.
// Here that is per-GPU CUDA streams with chunked host<->device copies overlapping the kernels,
// frame batches or row bands as the unit of work, and no collectives.
#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <tuple>
#include <vector>

#include <cuda_runtime.h>

#include "../../include/lanczos_b200.h"
#include "kernels.cuh"
#include "plan.h"

namespace lzb {
namespace {

thread_local std::string g_last_cuda_error;
thread_local lanczos_stats g_stats{};
thread_local lanczos_launch g_launch{};
std::atomic<bool> g_stats_enabled{false};

int cuda_fail(cudaError_t e, const char *what) {
    g_last_cuda_error = std::string(what) + ": " + cudaGetErrorString(e);
    return LANCZOS_ERR_CUDA;
}
#define CU(call)                                               \
    do {                                                       \
        cudaError_t e__ = (call);                              \
        if (e__ != cudaSuccess) return cuda_fail(e__, #call);  \
    } while (0)

struct DeviceGuard {
    int prev = -1;
    bool ok = false;
    explicit DeviceGuard(int dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        ok = cudaSetDevice(dev) == cudaSuccess;
    }
    ~DeviceGuard() {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

// Non-blocking streams of the host drivers, kept per device between calls (creating and destroying a stream
// costs tens of microseconds).  A lease synchronises its stream before handing it back, on every exit path,
// so no copy or kernel is still running on a scratch buffer when the buffer returns to its pool.
std::mutex g_stream_mutex;
std::map<int, std::vector<cudaStream_t>> g_idle_streams;
struct StreamLease {
    int device = -1;
    cudaStream_t s = nullptr;
    cudaError_t acquire(int dev) {
        device = dev;
        {
            std::lock_guard<std::mutex> l(g_stream_mutex);
            auto &v = g_idle_streams[dev];
            if (!v.empty()) {
                s = v.back();
                v.pop_back();
                return cudaSuccess;
            }
        }
        return cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking);
    }
    cudaError_t sync() { return s ? cudaStreamSynchronize(s) : cudaSuccess; }
    ~StreamLease() {
        if (!s) return;
        if (cudaStreamSynchronize(s) != cudaSuccess) {   // sticky error: do not reuse
            cudaStreamDestroy(s);
            return;
        }
        std::lock_guard<std::mutex> l(g_stream_mutex);
        g_idle_streams[device].push_back(s);
    }
    StreamLease() = default;
    StreamLease(const StreamLease &) = delete;
    StreamLease &operator=(const StreamLease &) = delete;
};

// Row-pitched copies between a caller's host image (pitch = the caller's) and a device scratch image whose
// pitch is the row size rounded up to 16 bytes (what the TMA kernels want).  Only the pixels of a row are
// touched on either side: padding bytes of the caller's buffer are neither read nor written.
long long scratch_pitch(long long row_bytes) { return (row_bytes + 15) / 16 * 16; }

// The host drivers own their device buffers, so they may run the kernels on a WIDENED image: input and output
// widths rounded up until a row is a whole number of 32-bit words (what the TMA kernels need), the extra input
// columns zero.  A zero column is the reference's dropped tap (full_TB.h:59: taps outside the row are skipped,
// no renormalisation) and every output column is computed independently of the others, so the original columns
// come out bit for bit; the extra output columns are never copied back.  The reference's own sample size
// (lanczos.h:13-14: 162 -> 486 pixels, planar) takes the specialised kernels this way.
// The extra output columns must not change which descriptors are accepted: when one of them fails the reference's
// float floor (LANCZOS_ERR_RATIO_FLOAT) the image is run at its own widths, as the device entry points would run it.
lanczos_desc widened(const lanczos_desc &r) {
    lanczos_desc d = r;            // resolved: scale_n / scale_d are explicit, so the ratio does not follow the new widths
    d.in_pitch = d.out_pitch = 0;
    const int q = d.channels == 4 ? 1 : (d.channels == 2 ? 2 : 4);
    const int out_w = (r.out_w + q - 1) / q * q;
    if (!float_floor_exact(r.out_w, out_w, r.scale_n, r.scale_d)) return d;
    d.in_w = (r.in_w + q - 1) / q * q;
    d.out_w = out_w;
    return d;
}
cudaError_t copy_rows(void *dst, long long dpitch, const void *src, long long spitch, long long row_bytes, long long rows,
                      cudaMemcpyKind kind, cudaStream_t s) {
    if (rows <= 0) return cudaSuccess;
    if (dpitch == row_bytes && spitch == row_bytes) return cudaMemcpyAsync(dst, src, (size_t)(row_bytes * rows), kind, s);
    return cudaMemcpy2DAsync(dst, (size_t)dpitch, src, (size_t)spitch, (size_t)row_bytes, (size_t)rows, kind, s);
}

// ---- host plans (tables only, no device memory), cached per geometry ---------------------------
using HostKey = std::tuple<int, int, int, int, int, int, int, int, unsigned>;
std::mutex g_host_plan_mutex;
std::map<HostKey, std::shared_ptr<const Plan>> g_host_plans;
constexpr unsigned kPlanFlagMask = LANCZOS_FLAG_NO_ALIAS;  // flags that change the tables

int get_host_plan(const lanczos_desc *desc, std::shared_ptr<const Plan> *out) {
    lanczos_desc r;
    int rc = resolve_desc(desc, &r);
    if (rc != LANCZOS_OK) return rc;
    HostKey key{r.in_w, r.in_h, r.out_w, r.out_h, r.channels, r.a, r.scale_n, r.scale_d, r.flags & kPlanFlagMask};
    {
        std::lock_guard<std::mutex> lock(g_host_plan_mutex);
        auto it = g_host_plans.find(key);
        if (it != g_host_plans.end()) {
            *out = it->second;
            return LANCZOS_OK;
        }
    }
    auto p = std::make_shared<Plan>();
    rc = build_plan(&r, p.get());   // O(out_w + out_h) libm calls: outside the lock
    if (rc != LANCZOS_OK) return rc;
    // plans are shared by callers with different row pitches: nothing may read the pitches of the first caller
    p->d.in_pitch = p->d.out_pitch = 0;
    std::lock_guard<std::mutex> lock(g_host_plan_mutex);
    auto ins = g_host_plans.emplace(key, p);
    *out = ins.first->second;
    return LANCZOS_OK;
}

// ---- device-resident plan -----------------------------------------------------------------
struct DevicePlan {
    std::shared_ptr<const Plan> host_ref;
    const Plan &host() const { return *host_ref; }
    std::mutex stats_mutex;   // the strict-sample counter is one per plan: calls that count take turns
    int device = 0;
    void *blob = nullptr;  // one allocation holding every table
    const int32_t *i0x = nullptr, *i0y = nullptr;
    const float *wfx = nullptr, *wfy = nullptr, *phase_w = nullptr;
    const double *wdx = nullptr, *wdy = nullptr;
    unsigned long long *strict_counter = nullptr;
    ~DevicePlan() {
        if (blob) {
            DeviceGuard g(device);
            cudaFree(blob);
        }
    }
};

using PlanKey = std::tuple<int, int, int, int, int, int, int, int, unsigned, int>;
std::mutex g_plan_mutex;
std::map<PlanKey, std::shared_ptr<DevicePlan>> g_plans;

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

int get_plan(const lanczos_desc *desc, int device, std::shared_ptr<DevicePlan> *out) {
    lanczos_desc r;
    int rc = resolve_desc(desc, &r);
    if (rc != LANCZOS_OK) return rc;
    PlanKey key{r.in_w, r.in_h, r.out_w, r.out_h, r.channels, r.a, r.scale_n, r.scale_d,
                r.flags & kPlanFlagMask, device};
    std::lock_guard<std::mutex> lock(g_plan_mutex);
    auto it = g_plans.find(key);
    if (it != g_plans.end()) {
        *out = it->second;
        return LANCZOS_OK;
    }
    auto dp = std::make_shared<DevicePlan>();
    dp->device = device;
    rc = get_host_plan(&r, &dp->host_ref);
    if (rc != LANCZOS_OK) return rc;
    const Plan &h = dp->host();
    // layout of the single device blob (each table 256-byte aligned)
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 256); return o; };
    const size_t o_wdx = take(h.x.wd.size() * 8), o_wdy = take(h.y.wd.size() * 8);
    const size_t o_wfx = take(h.x.wf.size() * 4), o_wfy = take(h.y.wf.size() * 4);
    const size_t o_i0x = take(h.x.i0.size() * 4), o_i0y = take(h.y.i0.size() * 4);
    const size_t o_ph = take(h.phase_w.size() * 4), o_cnt = take(8);
    std::vector<uint8_t> stage(off, 0);
    memcpy(&stage[o_wdx], h.x.wd.data(), h.x.wd.size() * 8);
    memcpy(&stage[o_wdy], h.y.wd.data(), h.y.wd.size() * 8);
    memcpy(&stage[o_wfx], h.x.wf.data(), h.x.wf.size() * 4);
    memcpy(&stage[o_wfy], h.y.wf.data(), h.y.wf.size() * 4);
    memcpy(&stage[o_i0x], h.x.i0.data(), h.x.i0.size() * 4);
    memcpy(&stage[o_i0y], h.y.i0.data(), h.y.i0.size() * 4);
    memcpy(&stage[o_ph], h.phase_w.data(), h.phase_w.size() * 4);
    CU(cudaMalloc(&dp->blob, off));
    CU(cudaMemcpy(dp->blob, stage.data(), off, cudaMemcpyHostToDevice));
    auto *b = (uint8_t *)dp->blob;
    dp->wdx = (const double *)(b + o_wdx);
    dp->wdy = (const double *)(b + o_wdy);
    dp->wfx = (const float *)(b + o_wfx);
    dp->wfy = (const float *)(b + o_wfy);
    dp->i0x = (const int32_t *)(b + o_i0x);
    dp->i0y = (const int32_t *)(b + o_i0y);
    dp->phase_w = (const float *)(b + o_ph);
    dp->strict_counter = (unsigned long long *)(b + o_cnt);
    g_plans[key] = dp;
    *out = dp;
    return LANCZOS_OK;
}

// ---- per-device scratch pool (host drivers only) -------------------------------------------
struct Pool {
    std::mutex m;
    std::vector<std::pair<void *, size_t>> free_list;
};
std::mutex g_pool_mutex;
std::map<int, std::unique_ptr<Pool>> g_pools;
Pool &pool_for(int device) {
    std::lock_guard<std::mutex> l(g_pool_mutex);
    auto &p = g_pools[device];
    if (!p) p.reset(new Pool);
    return *p;
}
struct Scratch {  // RAII device buffer from the pool (current device must be `device`)
    int device;
    void *p = nullptr;
    size_t cap = 0;
    Scratch(int dev, size_t bytes) : device(dev) {
        bytes = std::max<size_t>(bytes, 256);
        Pool &pl = pool_for(dev);
        {
            std::lock_guard<std::mutex> l(pl.m);
            size_t best = (size_t)-1, bi = 0;
            for (size_t i = 0; i < pl.free_list.size(); i++)
                if (pl.free_list[i].second >= bytes && pl.free_list[i].second < best) best = pl.free_list[i].second, bi = i;
            if (best != (size_t)-1) {
                p = pl.free_list[bi].first;
                cap = best;
                pl.free_list.erase(pl.free_list.begin() + bi);
                return;
            }
        }
        if (cudaMalloc(&p, bytes) == cudaSuccess) cap = bytes; else p = nullptr;
    }
    ~Scratch() {
        if (!p) return;
        Pool &pl = pool_for(device);
        std::lock_guard<std::mutex> l(pl.m);
        pl.free_list.emplace_back(p, cap);
    }
    Scratch(const Scratch &) = delete;
    Scratch &operator=(const Scratch &) = delete;
};

// ---- core launch ----------------------------------------------------------------------------
constexpr int kMaxGridFrames = 65535;

// the first main launch of a call (main_launches is counted by the caller)
void set_launch(const LaunchShape &sh) {
    g_launch.grid_x = sh.grid_x;
    g_launch.grid_y = sh.grid_y;
    g_launch.grid_z = sh.grid_z;
    g_launch.seg_periods = sh.seg_periods;
    g_launch.chunk_rows = sh.chunk_rows;
    g_launch.resident_ctas = sh.resident_ctas;
}

int run_device(const DevicePlan &dp, unsigned flags, const uint8_t *d_in, uint8_t *d_out, int n_frames,
               long long in_frame_stride, long long out_frame_stride, int out_row0, int out_rows,
               int in_row0, int in_rows, long long in_pitch, long long out_pitch, cudaStream_t s) {
    const Plan &h = dp.host();
    KParams p{};
    p.in = d_in;
    p.out = d_out;
    p.in_pitch = in_pitch;
    p.out_pitch = out_pitch;
    p.in_frame_stride = in_frame_stride;
    p.out_frame_stride = out_frame_stride;
    p.n_frames = n_frames;
    p.in_w = h.d.in_w; p.in_h = h.d.in_h; p.out_w = h.d.out_w; p.out_h = h.d.out_h;
    p.channels = h.d.channels; p.a = h.d.a; p.taps = h.taps;
    p.scale_n = h.d.scale_n; p.scale_d = h.d.scale_d;
    p.out_row0 = out_row0; p.out_rows = out_rows; p.in_row0 = in_row0; p.in_rows = in_rows;
    p.i0x = dp.i0x; p.wfx = dp.wfx; p.wdx = dp.wdx;
    p.i0y = dp.i0y; p.wfy = dp.wfy; p.wdy = dp.wdy;
    p.phase_w = dp.phase_w;
    p.guard = h.guard;
    p.guard_asc = h.guard_asc;
    p.guard_outer = h.guard_outer;
    p.alias_rows = h.alias_rows; p.alias_top_row = h.alias_top_row; p.alias_in_rows = h.alias_in_rows;
    p.flags = flags;
    const bool count = g_stats_enabled.load(std::memory_order_relaxed);
    p.strict_counter = count ? dp.strict_counter : nullptr;
    g_stats = lanczos_stats{};
    g_launch = lanczos_launch{};
    if (n_frames <= 0 || out_rows <= 0) return LANCZOS_OK;
    // counting calls are synchronous and take turns on the plan's counter (several host threads or streams may share a plan)
    std::unique_lock<std::mutex> stats_lock;
    if (count) {
        stats_lock = std::unique_lock<std::mutex>(const_cast<DevicePlan &>(dp).stats_mutex);
        CU(cudaMemsetAsync(dp.strict_counter, 0, 8, s));
    }

    // CUDA caps a grid's y and z dimensions at 65,535 (frames are gridDim.z of the main kernels and gridDim.y of the
    // alias-rows kernel): larger batches run as consecutive frame groups, each with its own tensor map and plan
    for (int g0 = 0; g0 < n_frames; g0 += kMaxGridFrames) {
        p.in = d_in + (long long)g0 * in_frame_stride;
        p.out = d_out + (long long)g0 * out_frame_stride;
        p.n_frames = std::min(kMaxGridFrames, n_frames - g0);
        int kid = 0, alias_done = 0;
        int frc = -1;
        LaunchShape shape;
        if (!(flags & LANCZOS_FLAG_GENERIC_KERNEL)) {
            FastHostTables t{h.phase_w.data(), h.phase_wd.data(), h.align_k.data(), h.x.aligned_exact ? 1 : 0,
                             h.y.aligned_exact ? 1 : 0, h.x.uniform_phase ? 1 : 0, h.y.uniform_phase ? 1 : 0, h.x.i0.data(),
                             h.p0_chain_ok ? h.p0_chain : nullptr};
            frc = launch_v6(p, t, &kid, &alias_done, &shape, s);
            if (frc < 0) frc = launch_dyn(p, t, &kid, &shape, s);
        }
        if (frc > 0) return cuda_fail((cudaError_t)frc, "specialised kernel launch");
        cudaError_t e = cudaSuccess;
        if (frc < 0) {
            kid = 0;
            e = (cudaError_t)launch_generic(p, &shape, s);
        }
        if (e != cudaSuccess) return cuda_fail(e, "launch_generic");
        g_stats.kernel_launches++;
        g_stats.kernel_id = kid;
        if (g0 == 0) set_launch(shape);
        g_launch.main_launches++;
        if (h.alias_rows > 0 && out_row0 < h.alias_rows && alias_done) {
            g_stats.alias_rows = std::min(h.alias_rows, out_row0 + out_rows) - out_row0;
        } else if (h.alias_rows > 0 && out_row0 < h.alias_rows) {
            e = (cudaError_t)launch_alias_rows(p, s);
            if (e != cudaSuccess) return cuda_fail(e, "launch_alias_rows");
            g_stats.kernel_launches++;
            g_stats.alias_rows = std::min(h.alias_rows, out_row0 + out_rows) - out_row0;
        }
    }
    if (count) {
        unsigned long long c = 0;
        CU(cudaMemcpyAsync(&c, dp.strict_counter, 8, cudaMemcpyDeviceToHost, s));
        CU(cudaStreamSynchronize(s));
        g_stats.strict_samples = (int64_t)c;
    }
    return LANCZOS_OK;
}

int check_band(const Plan &h, int out_row0, int out_rows, int in_row0, int in_rows) {
    if (out_row0 < 0 || out_rows < 0 || out_row0 + out_rows > h.d.out_h) return LANCZOS_ERR_BAND;
    if (out_rows == 0) return LANCZOS_OK;
    // the supplied rows must be rows of the image: a kernel indexes them as (row - in_row0) * pitch
    if (in_row0 < 0 || in_rows < 0 || in_row0 + in_rows > h.d.in_h) return LANCZOS_ERR_BAND;
    int need0, needn;
    band_rows(h, out_row0, out_rows, &need0, &needn);
    if (in_row0 > need0 || in_row0 + in_rows < need0 + needn) return LANCZOS_ERR_BAND;
    return LANCZOS_OK;
}

}  // namespace
}  // namespace lzb

using namespace lzb;

extern "C" {

int lanczos_b200_abi_version(void) { return LANCZOS_B200_ABI_VERSION; }

const char *lanczos_b200_strerror(int code) {
    switch (code) {
        case LANCZOS_OK: return "ok";
        case LANCZOS_ERR_NULL: return "null descriptor or buffer";
        case LANCZOS_ERR_DIMS: return "bad dimensions or pitches";
        case LANCZOS_ERR_CHANNELS: return "channels must be 1..4";
        case LANCZOS_ERR_TAPS: return "a (taps per side) must be 1..4";
        case LANCZOS_ERR_RATIO: return "scale ratio must be a positive upscale N/D >= 1";
        case LANCZOS_ERR_RATIO_FLOAT: return "floor((double)xx/SCALE) differs from floor(xx*D/N) for this ratio and size";
        case LANCZOS_ERR_BAND: return "row band outside the image or input rows not supplied";
        case LANCZOS_ERR_CUDA: return "CUDA error";
        case LANCZOS_ERR_NOMEM: return "out of memory";
        case LANCZOS_ERR_ALIGN: return "unsupported layout for this entry point";
        default: return "unknown error";
    }
}

const char *lanczos_b200_last_cuda_error(void) { return g_last_cuda_error.c_str(); }

void lanczos_b200_enable_stats(int on) { g_stats_enabled.store(on != 0, std::memory_order_relaxed); }

int lanczos_b200_get_stats(lanczos_stats *out) {
    if (!out) return LANCZOS_ERR_NULL;
    *out = g_stats;
    return LANCZOS_OK;
}

int lanczos_b200_get_launch(lanczos_launch *out) {
    if (!out) return LANCZOS_ERR_NULL;
    *out = g_launch;
    return LANCZOS_OK;
}

void lanczos_b200_clear_plans(void) {
    {
        std::lock_guard<std::mutex> lock(g_plan_mutex);
        g_plans.clear();
    }
    {
        std::lock_guard<std::mutex> lock(g_host_plan_mutex);
        g_host_plans.clear();
    }
    std::lock_guard<std::mutex> l(g_pool_mutex);
    for (auto &kv : g_pools) {
        DeviceGuard g(kv.first);
        std::lock_guard<std::mutex> l2(kv.second->m);
        for (auto &b : kv.second->free_list) cudaFree(b.first);
        kv.second->free_list.clear();
    }
}

int lanczos_b200_reduce_ratio(int32_t out_len, int32_t in_len, int32_t *scale_n, int32_t *scale_d) {
    if (!scale_n || !scale_d) return LANCZOS_ERR_NULL;
    if (out_len < 1 || in_len < 1) return LANCZOS_ERR_DIMS;
    int a = out_len, b = in_len;
    while (b) { int t = a % b; a = b; b = t; }  // stb.cpp:9-12
    *scale_n = out_len / a;
    *scale_d = in_len / a;
    return LANCZOS_OK;
}

int lanczos_b200_resolve(const lanczos_desc *desc, lanczos_desc *resolved) { return resolve_desc(desc, resolved); }

double lanczos_b200_kernel(double x, int32_t a) { return ref_kernel(x, a); }

int lanczos_b200_phase_table(const lanczos_desc *desc, float *weights, int32_t capacity_floats) {
    if (!desc) return LANCZOS_ERR_NULL;
    Plan p;
    // only the table is wanted: shrink the image so the per-coordinate tables stay tiny
    lanczos_desc d = *desc;
    int rc = resolve_desc(desc, &d);
    if (rc != LANCZOS_OK) return rc;
    lanczos_desc small = d;
    small.in_w = small.in_h = d.scale_d;
    small.out_w = small.out_h = d.scale_n;
    small.in_pitch = small.out_pitch = 0;
    rc = build_plan(&small, &p);
    if (rc != LANCZOS_OK) return rc;
    const int need = d.scale_n * 2 * d.a;
    if (weights) {
        if (capacity_floats < need) return LANCZOS_ERR_DIMS;
        memcpy(weights, p.phase_w.data(), sizeof(float) * need);
    }
    return d.scale_n;
}

int lanczos_b200_phase0_chain(const lanczos_desc *desc, float *consts) {
    if (!desc || !consts) return LANCZOS_ERR_NULL;
    lanczos_desc d = *desc;
    int rc = resolve_desc(desc, &d);
    if (rc != LANCZOS_OK) return rc;
    lanczos_desc small = d;
    small.in_w = small.in_h = d.scale_d;
    small.out_w = small.out_h = d.scale_n;
    small.in_pitch = small.out_pitch = 0;
    Plan p;
    rc = build_plan(&small, &p);
    if (rc != LANCZOS_OK) return rc;
    memcpy(consts, p.p0_chain, sizeof(p.p0_chain));
    return p.p0_chain_ok ? 1 : 0;
}

int lanczos_b200_alias_rows(const lanczos_desc *desc) {
    if (!desc) return LANCZOS_ERR_NULL;
    std::shared_ptr<const Plan> p;
    int rc = get_host_plan(desc, &p);
    if (rc != LANCZOS_OK) return rc;
    return p->alias_rows;
}

int lanczos_b200_band_input_rows(const lanczos_desc *desc, int32_t out_row0, int32_t out_rows,
                                 int32_t *in_row0, int32_t *in_rows) {
    if (!desc || !in_row0 || !in_rows) return LANCZOS_ERR_NULL;
    std::shared_ptr<const Plan> p;
    int rc = get_host_plan(desc, &p);
    if (rc != LANCZOS_OK) return rc;
    if (out_row0 < 0 || out_rows < 1 || out_row0 + out_rows > p->d.out_h) return LANCZOS_ERR_BAND;
    int a, b;
    band_rows(*p, out_row0, out_rows, &a, &b);
    *in_row0 = a;
    *in_rows = b;
    return LANCZOS_OK;
}

int lanczos_b200_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}

void *lanczos_b200_host_alloc(size_t bytes) {
    void *p = nullptr;
    if (cudaMallocHost(&p, bytes ? bytes : 1) != cudaSuccess) return nullptr;
    return p;
}
void lanczos_b200_host_free(void *p) {
    if (p) cudaFreeHost(p);
}
void *lanczos_b200_device_alloc(int device, size_t bytes) {
    DeviceGuard g(device);
    if (!g.ok) return nullptr;
    void *p = nullptr;
    if (cudaMalloc(&p, bytes ? bytes : 1) != cudaSuccess) return nullptr;
    return p;
}
void lanczos_b200_device_free(int device, void *p) {
    if (!p) return;
    DeviceGuard g(device);
    cudaFree(p);
}
int lanczos_b200_memcpy_h2d(int device, void *d_dst, const void *h_src, size_t bytes) {
    DeviceGuard g(device);
    if (!g.ok) return cuda_fail(cudaErrorInvalidDevice, "cudaSetDevice");
    CU(cudaMemcpy(d_dst, h_src, bytes, cudaMemcpyHostToDevice));
    return LANCZOS_OK;
}
int lanczos_b200_memcpy_d2h(int device, void *h_dst, const void *d_src, size_t bytes) {
    DeviceGuard g(device);
    if (!g.ok) return cuda_fail(cudaErrorInvalidDevice, "cudaSetDevice");
    CU(cudaMemcpy(h_dst, d_src, bytes, cudaMemcpyDeviceToHost));
    return LANCZOS_OK;
}
int lanczos_b200_synchronize(int device) {
    DeviceGuard g(device);
    if (!g.ok) return cuda_fail(cudaErrorInvalidDevice, "cudaSetDevice");
    CU(cudaDeviceSynchronize());
    return LANCZOS_OK;
}

// ---- device-buffer entry points -------------------------------------------------------------

int lanczos_b200_upscale_batch(const lanczos_desc *desc, const uint8_t *d_in, uint8_t *d_out,
                               int32_t n_frames, int64_t in_frame_stride, int64_t out_frame_stride,
                               int device, void *cuda_stream) {
    if (!desc || !d_in || !d_out) return LANCZOS_ERR_NULL;
    if (n_frames < 0) return LANCZOS_ERR_DIMS;
    DeviceGuard g(device);
    if (!g.ok) return cuda_fail(cudaErrorInvalidDevice, "cudaSetDevice");
    std::shared_ptr<DevicePlan> dp;
    int rc = get_plan(desc, device, &dp);
    if (rc != LANCZOS_OK) return rc;
    const lanczos_desc &r = dp->host().d;
    lanczos_desc user;
    resolve_desc(desc, &user);  // user pitches (plans are shared across pitches)
    if (in_frame_stride == 0) in_frame_stride = user.in_pitch * r.in_h;
    if (out_frame_stride == 0) out_frame_stride = user.out_pitch * r.out_h;
    return run_device(*dp, desc->flags, d_in, d_out, n_frames, in_frame_stride, out_frame_stride, 0,
                      r.out_h, 0, r.in_h, user.in_pitch, user.out_pitch, (cudaStream_t)cuda_stream);
}

int lanczos_b200_upscale(const lanczos_desc *desc, const uint8_t *d_in, uint8_t *d_out, int device,
                         void *cuda_stream) {
    return lanczos_b200_upscale_batch(desc, d_in, d_out, 1, 0, 0, device, cuda_stream);
}

int lanczos_b200_upscale_planar(const lanczos_desc *desc, const uint8_t *d_in, uint8_t *d_out, int32_t n_frames,
                                int64_t in_plane_stride, int64_t out_plane_stride, int device, void *cuda_stream) {
    if (!desc || !d_in || !d_out) return LANCZOS_ERR_NULL;
    if (n_frames < 0) return LANCZOS_ERR_DIMS;
    if (desc->channels < 1 || desc->channels > 4) return LANCZOS_ERR_CHANNELS;
    const int64_t planes = (int64_t)n_frames * desc->channels;
    if (planes > INT32_MAX) return LANCZOS_ERR_DIMS;
    // a plane is a one-channel frame: the reference's own loop is per channel, rows then columns (full_TB.h:83-95)
    lanczos_desc plane = *desc;
    plane.channels = 1;
    return lanczos_b200_upscale_batch(&plane, d_in, d_out, (int32_t)planes, in_plane_stride, out_plane_stride,
                                      device, cuda_stream);
}

int lanczos_b200_upscale_band(const lanczos_desc *desc, const uint8_t *d_in_band, uint8_t *d_out_band,
                              int32_t out_row0, int32_t out_rows, int32_t in_row0, int32_t in_rows,
                              int device, void *cuda_stream) {
    if (!desc || !d_in_band || !d_out_band) return LANCZOS_ERR_NULL;
    DeviceGuard g(device);
    if (!g.ok) return cuda_fail(cudaErrorInvalidDevice, "cudaSetDevice");
    std::shared_ptr<DevicePlan> dp;
    int rc = get_plan(desc, device, &dp);
    if (rc != LANCZOS_OK) return rc;
    rc = check_band(dp->host(), out_row0, out_rows, in_row0, in_rows);
    if (rc != LANCZOS_OK) return rc;
    lanczos_desc user;
    resolve_desc(desc, &user);
    return run_device(*dp, desc->flags, d_in_band, d_out_band, 1, 0, 0, out_row0, out_rows, in_row0,
                      in_rows, user.in_pitch, user.out_pitch, (cudaStream_t)cuda_stream);
}

// ---- fixed-point HLS mode --------------------------------------------------------------------

int lanczos_b200_hls_lut(int32_t a, int32_t scale_n, int32_t bit_precision, int32_t *lut, int32_t capacity) {
    if (!lut) return LANCZOS_ERR_NULL;
    if (a < 1 || a > kMaxTaps / 2) return LANCZOS_ERR_TAPS;
    if (scale_n < 1 || a * scale_n > 127) return LANCZOS_ERR_RATIO;   // kernel_t(i) wraps for i >= 128
    if (bit_precision < 1 || bit_precision > 12 || capacity < a * scale_n + 1) return LANCZOS_ERR_DIMS;
    for (int i = 0; i < a * scale_n; i++) {
        // kernel.cpp:42: argument (kernel_t)i/SCALE_N truncated to BP bits, value truncated to BP bits (AP_TRN)
        const double x = std::floor((double)i * (1 << bit_precision) / scale_n) / (1 << bit_precision);
        lut[i] = (int32_t)std::floor(ref_kernel(x, a) * (1 << bit_precision));
    }
    lut[a * scale_n] = 0;   // kernel.cpp:44
    return LANCZOS_OK;
}

int lanczos_b200_upscale_hls(const lanczos_desc *desc, const uint8_t *d_in, uint8_t *d_out, int32_t bit_precision,
                             int32_t n_frames, int64_t in_frame_stride, int64_t out_frame_stride, int device,
                             void *cuda_stream) {
    if (!desc || !d_in || !d_out) return LANCZOS_ERR_NULL;
    if (n_frames < 0) return LANCZOS_ERR_DIMS;
    lanczos_desc r;
    int rc = resolve_desc(desc, &r);
    if (rc != LANCZOS_OK) return rc;
    if (r.scale_d != 1) return LANCZOS_ERR_RATIO;   // the BP-bit step condition drifts for other ratios
    int32_t lut[128];
    rc = lanczos_b200_hls_lut(r.a, r.scale_n, bit_precision, lut, 128);
    if (rc != LANCZOS_OK) return rc;
    DeviceGuard g(device);
    if (!g.ok) return cuda_fail(cudaErrorInvalidDevice, "cudaSetDevice");
    if (in_frame_stride == 0) in_frame_stride = r.in_pitch * r.in_h;
    if (out_frame_stride == 0) out_frame_stride = r.out_pitch * r.out_h;
    g_stats = lanczos_stats{};
    g_launch = lanczos_launch{};
    for (int g0 = 0; g0 < n_frames; g0 += kMaxGridFrames) {   // frame groups, as in run_device
        int kid = 100;
        LaunchShape shape;
        cudaError_t e = (cudaError_t)launch_hls(d_in + (long long)g0 * in_frame_stride, d_out + (long long)g0 * out_frame_stride,
                                                r.in_pitch, r.out_pitch, in_frame_stride, out_frame_stride,
                                                std::min(kMaxGridFrames, n_frames - g0), r.in_w, r.in_h, r.out_w, r.out_h,
                                                r.channels, r.a, r.scale_n, bit_precision, lut, &kid, &shape,
                                                (cudaStream_t)cuda_stream);
        if (e != cudaSuccess) return cuda_fail(e, "launch_hls");
        g_stats.kernel_launches++;
        g_stats.kernel_id = kid;
        if (g0 == 0) set_launch(shape);
        g_launch.main_launches++;
    }
    return LANCZOS_OK;
}

// ---- host-buffer drivers --------------------------------------------------------------------

int lanczos_b200_upscale_host(const lanczos_desc *desc, const uint8_t *h_in, uint8_t *h_out,
                              int32_t n_frames, int64_t in_frame_stride, int64_t out_frame_stride,
                              int device, int32_t n_streams) {
    if (!desc || !h_in || !h_out) return LANCZOS_ERR_NULL;
    if (n_frames < 0) return LANCZOS_ERR_DIMS;
    DeviceGuard g(device);
    if (!g.ok) return cuda_fail(cudaErrorInvalidDevice, "cudaSetDevice");
    lanczos_desc user;
    int rc = resolve_desc(desc, &user);
    if (rc != LANCZOS_OK) return rc;
    const lanczos_desc wide = widened(user);
    const bool is_wide = wide.in_w != user.in_w || wide.out_w != user.out_w;
    std::shared_ptr<DevicePlan> dp;
    rc = get_plan(&wide, device, &dp);
    if (rc != LANCZOS_OK) return rc;
    const Plan &h = dp->host();
    const long long in_row = (long long)user.in_w * user.channels, out_row = (long long)user.out_w * user.channels;
    const long long d_in_pitch = scratch_pitch((long long)wide.in_w * wide.channels), d_out_pitch = scratch_pitch((long long)wide.out_w * wide.channels);
    if (in_frame_stride == 0) in_frame_stride = user.in_pitch * h.d.in_h;
    if (out_frame_stride == 0) out_frame_stride = user.out_pitch * h.d.out_h;
    if (n_streams < 1) n_streams = 3;
    n_streams = std::min(n_streams, 8);

    // Work items: whole frames when there are several, otherwise row bands of the single frame,
    // so that host->device, kernel and device->host of different items overlap.
    struct Item { int frame, out_row0, out_rows, in_row0, in_rows; };
    std::vector<Item> items;
    if (n_frames >= 2 * n_streams) {
        for (int f = 0; f < n_frames; f++) items.push_back({f, 0, h.d.out_h, 0, h.d.in_h});
    } else {
        const int bands = std::max(1, std::min(h.d.out_h / 64, 2 * n_streams));
        for (int f = 0; f < n_frames; f++)
            for (int b = 0; b < bands; b++) {
                const int r0 = (int)((long long)h.d.out_h * b / bands), r1 = (int)((long long)h.d.out_h * (b + 1) / bands);
                if (r1 <= r0) continue;
                Item it{f, r0, r1 - r0, 0, 0};
                band_rows(h, r0, r1 - r0, &it.in_row0, &it.in_rows);
                items.push_back(it);
            }
    }
    size_t max_in = 0, max_out = 0;
    for (auto &it : items) {
        max_in = std::max(max_in, (size_t)(it.in_rows * d_in_pitch));
        max_out = std::max(max_out, (size_t)(it.out_rows * d_out_pitch));
    }
    n_streams = std::max(1, std::min<int>(n_streams, (int)items.size()));
    // declaration order matters: the leases are destroyed (= synchronised) before the scratch buffers are released
    std::vector<std::unique_ptr<Scratch>> bin(n_streams), bout(n_streams);
    std::vector<StreamLease> streams(n_streams);
    for (int i = 0; i < n_streams; i++) {
        CU(streams[i].acquire(device));
        bin[i].reset(new Scratch(device, max_in));
        bout[i].reset(new Scratch(device, max_out));
        if (!bin[i]->p || !bout[i]->p) return LANCZOS_ERR_NOMEM;
        if (is_wide) CU(cudaMemsetAsync(bin[i]->p, 0, max_in, streams[i].s));   // the extra columns stay zero: only pixels are copied in
    }
    int64_t launches = 0;
    for (size_t k = 0; k < items.size(); k++) {
        const Item &it = items[k];
        const int si = (int)(k % n_streams);
        cudaStream_t s = streams[si].s;
        const uint8_t *src = h_in + it.frame * in_frame_stride + (long long)it.in_row0 * user.in_pitch;
        uint8_t *dst = h_out + it.frame * out_frame_stride + (long long)it.out_row0 * user.out_pitch;
        CU(copy_rows(bin[si]->p, d_in_pitch, src, user.in_pitch, in_row, it.in_rows, cudaMemcpyHostToDevice, s));
        rc = run_device(*dp, desc->flags, (const uint8_t *)bin[si]->p, (uint8_t *)bout[si]->p, 1, 0, 0,
                        it.out_row0, it.out_rows, it.in_row0, it.in_rows, d_in_pitch, d_out_pitch, s);
        launches += g_stats.kernel_launches;
        if (rc != LANCZOS_OK) return rc;
        CU(copy_rows(dst, user.out_pitch, bout[si]->p, d_out_pitch, out_row, it.out_rows, cudaMemcpyDeviceToHost, s));
    }
    for (int i = 0; i < n_streams; i++) CU(streams[i].sync());
    g_stats.kernel_launches = launches;
    return LANCZOS_OK;
}

int lanczos_b200_upscale_host_bands(const lanczos_desc *desc, const uint8_t *h_in, uint8_t *h_out,
                                    const int32_t *devices, int32_t n_devices) {
    if (!desc || !h_in || !h_out || !devices) return LANCZOS_ERR_NULL;
    if (n_devices < 1) return LANCZOS_ERR_DIMS;
    lanczos_desc user;
    int rc = resolve_desc(desc, &user);
    if (rc != LANCZOS_OK) return rc;
    const lanczos_desc wide = widened(user);
    const bool is_wide = wide.in_w != user.in_w || wide.out_w != user.out_w;
    const long long in_row = (long long)user.in_w * user.channels, out_row = (long long)user.out_w * user.channels;
    const long long d_in_pitch = scratch_pitch((long long)wide.in_w * wide.channels), d_out_pitch = scratch_pitch((long long)wide.out_w * wide.channels);
    std::vector<int> rcs(n_devices, LANCZOS_OK);
    std::vector<std::string> errs(n_devices);
    std::vector<int64_t> launches(n_devices, 0);
    std::vector<std::thread> workers;
    for (int gidx = 0; gidx < n_devices; gidx++) {
        workers.emplace_back([&, gidx]() {
            const int dev = devices[gidx];
            const int r0 = (int)((long long)user.out_h * gidx / n_devices);
            const int r1 = (int)((long long)user.out_h * (gidx + 1) / n_devices);
            if (r1 <= r0) return;
            auto body = [&]() -> int {
                DeviceGuard g(dev);
                if (!g.ok) return cuda_fail(cudaErrorInvalidDevice, "cudaSetDevice");
                std::shared_ptr<DevicePlan> dp;
                int rc2 = get_plan(&wide, dev, &dp);
                if (rc2 != LANCZOS_OK) return rc2;
                int in0, inn;
                band_rows(dp->host(), r0, r1 - r0, &in0, &inn);
                Scratch bin(dev, (size_t)(inn * d_in_pitch)), bout(dev, (size_t)((r1 - r0) * d_out_pitch));
                if (!bin.p || !bout.p) return LANCZOS_ERR_NOMEM;
                StreamLease st;   // after the scratch buffers: synchronised before they are released
                CU(st.acquire(dev));
                if (is_wide) CU(cudaMemsetAsync(bin.p, 0, (size_t)(inn * d_in_pitch), st.s));
                CU(copy_rows(bin.p, d_in_pitch, h_in + (long long)in0 * user.in_pitch, user.in_pitch, in_row, inn,
                             cudaMemcpyHostToDevice, st.s));
                rc2 = run_device(*dp, desc->flags, (const uint8_t *)bin.p, (uint8_t *)bout.p, 1, 0, 0, r0,
                                 r1 - r0, in0, inn, d_in_pitch, d_out_pitch, st.s);
                launches[gidx] = g_stats.kernel_launches;
                if (rc2 != LANCZOS_OK) return rc2;
                CU(copy_rows(h_out + (long long)r0 * user.out_pitch, user.out_pitch, bout.p, d_out_pitch, out_row, r1 - r0,
                             cudaMemcpyDeviceToHost, st.s));
                CU(st.sync());
                return LANCZOS_OK;
            };
            rcs[gidx] = body();
            errs[gidx] = g_last_cuda_error;
        });
    }
    for (auto &w : workers) w.join();
    g_stats = lanczos_stats{};
    for (int i = 0; i < n_devices; i++) {
        g_stats.kernel_launches += launches[i];
        if (rcs[i] != LANCZOS_OK) {
            g_last_cuda_error = errs[i];
            return rcs[i];
        }
    }
    return LANCZOS_OK;
}

int lanczos_b200_expected(const lanczos_desc *desc, const uint8_t *h_in_planar, uint8_t *h_out_planar,
                          int device) {
    if (!desc || !h_in_planar || !h_out_planar) return LANCZOS_ERR_NULL;
    lanczos_desc d = *desc;
    d.in_pitch = d.out_pitch = 0;  // planar arrays are dense (full_TB.h:20-21)
    lanczos_desc r;
    int rc = resolve_desc(&d, &r);
    if (rc != LANCZOS_OK) return rc;
    DeviceGuard g(device);
    if (!g.ok) return cuda_fail(cudaErrorInvalidDevice, "cudaSetDevice");
    // planes stay planes: each one is upscaled as a one-channel frame (no interleaving round trip); on the device
    // the rows of a plane are padded to 16 bytes so that odd widths keep the TMA kernels
    const long long planes = r.channels;
    lanczos_desc plane = r;
    plane.channels = 1;
    const lanczos_desc wide = widened(plane);               // one-channel planes: widths rounded up to 4 pixels
    const long long d_in_pitch = scratch_pitch(wide.in_w), d_out_pitch = scratch_pitch(wide.out_w);
    d = wide;
    d.channels = r.channels;
    d.in_pitch = d_in_pitch;
    d.out_pitch = d_out_pitch;
    Scratch pin(device, (size_t)(d_in_pitch * r.in_h * planes)), pout(device, (size_t)(d_out_pitch * r.out_h * planes));
    if (!pin.p || !pout.p) return LANCZOS_ERR_NOMEM;
    StreamLease st;
    CU(st.acquire(device));
    if (wide.in_w != r.in_w) CU(cudaMemsetAsync(pin.p, 0, (size_t)(d_in_pitch * r.in_h * planes), st.s));
    CU(copy_rows(pin.p, d_in_pitch, h_in_planar, r.in_w, r.in_w, (long long)r.in_h * planes, cudaMemcpyHostToDevice, st.s));
    rc = lanczos_b200_upscale_planar(&d, (const uint8_t *)pin.p, (uint8_t *)pout.p, 1, 0, 0, device, st.s);
    if (rc != LANCZOS_OK) return rc;
    CU(copy_rows(h_out_planar, r.out_w, pout.p, d_out_pitch, r.out_w, (long long)r.out_h * planes, cudaMemcpyDeviceToHost, st.s));
    CU(st.sync());
    return LANCZOS_OK;
}

int lanczos_b200_stream(const lanczos_desc *desc, const uint32_t *h_in_words, uint32_t *h_out_words, int device) {
    if (!desc || !h_in_words || !h_out_words) return LANCZOS_ERR_NULL;
    if (desc->channels != 3) return LANCZOS_ERR_ALIGN;
    lanczos_desc d = *desc;
    d.in_pitch = d.out_pitch = 0;   // a stream has no row padding (lanczos.cpp:56-62)
    DeviceGuard g(device);
    if (!g.ok) return cuda_fail(cudaErrorInvalidDevice, "cudaSetDevice");
    std::shared_ptr<DevicePlan> dp;
    int rc = get_plan(&d, device, &dp);
    if (rc != LANCZOS_OK) return rc;
    lanczos_desc r;
    resolve_desc(&d, &r);           // dense pitches of THIS call: cached plans carry none
    const long long n_in = (long long)r.in_w * r.in_h, n_out = (long long)r.out_w * r.out_h;
    Scratch win(device, n_in * 4), iin(device, n_in * 3), iout(device, n_out * 3), wout(device, n_out * 4);
    if (!win.p || !iin.p || !iout.p || !wout.p) return LANCZOS_ERR_NOMEM;
    StreamLease st;
    CU(st.acquire(device));
    CU(cudaMemcpyAsync(win.p, h_in_words, n_in * 4, cudaMemcpyHostToDevice, st.s));
    CU((cudaError_t)launch_words_to_rgb((const uint32_t *)win.p, (uint8_t *)iin.p, n_in, st.s));
    rc = run_device(*dp, d.flags, (const uint8_t *)iin.p, (uint8_t *)iout.p, 1, 0, 0, 0, r.out_h, 0, r.in_h,
                    r.in_pitch, r.out_pitch, st.s);
    if (rc != LANCZOS_OK) return rc;
    const int64_t launches = g_stats.kernel_launches + 2;
    CU((cudaError_t)launch_rgb_to_words((const uint8_t *)iout.p, (uint32_t *)wout.p, n_out, st.s));
    CU(cudaMemcpyAsync(h_out_words, wout.p, n_out * 4, cudaMemcpyDeviceToHost, st.s));
    CU(st.sync());
    g_stats.kernel_launches = launches;
    return LANCZOS_OK;
}

}  // extern "C"
