// extern "C" shim of include/b200rt.h: argument checking, device residency, launches. No compute happens on the host.
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <memory>
#include <new>
#include <string>
#include <thread>
#include <type_traits>
#include <vector>

#include <cuda_runtime.h>

#include "../../include/b200rt.h"
#include "bvh_build.h"
#include "device_types.h"
#include "kernels.h"
#include "obj_ingest.h"

using namespace b200rt;

struct b200rt_obj { ParsedObjArrays a; };
struct b200rt_hdr { std::vector<float> rgb; int w = 0, h = 0; };

struct b200rt_bvh { FlatBVH flat; };

// Owners of the CUDA resources the library keeps: each releases what it holds when it is destroyed or replaced, so an object or a call
// that fails halfway frees everything it had made. Device memory is released under whatever device is current, so an owner is
// destroyed inside the DeviceScope of the device it was allocated on.
struct DeviceFree { void operator()(void* p) const { cudaFree(p); } };
struct PinnedFree { void operator()(void* p) const { cudaFreeHost(p); } };
struct StreamDestroy { void operator()(cudaStream_t st) const { cudaStreamDestroy(st); } };
struct EventDestroy { void operator()(cudaEvent_t ev) const { cudaEventDestroy(ev); } };
using DevPtr = std::unique_ptr<void, DeviceFree>;
using PinnedPtr = std::unique_ptr<void, PinnedFree>;
using Stream = std::unique_ptr<std::remove_pointer_t<cudaStream_t>, StreamDestroy>;
using Event = std::unique_ptr<std::remove_pointer_t<cudaEvent_t>, EventDestroy>;

// A device array of T, grown on demand; its contents do not survive a grow. grow() frees the old array before it allocates (peak device
// memory never holds both) and records the capacity only once the allocation has succeeded, so after a failure it holds nothing.
template <typename T>
struct DevArray
{
    DevPtr mem;
    size_t cap = 0;
    T* get() const { return static_cast<T*>(mem.get()); }
    cudaError_t grow(size_t n)
    {
        if (n <= cap) return cudaSuccess;
        mem.reset(); cap = 0;
        void* p = nullptr;
        const cudaError_t e = cudaMalloc(&p, n * sizeof(T));
        if (e == cudaSuccess) { mem.reset(p); cap = n; }
        return e;
    }
};

struct b200rt_scene
{
    int device = 0;
    SceneDev dev{};
    b200rt_bvh_info info{};
    size_t bytes = 0;
    std::vector<DevPtr> allocs;           // the scene's uploads and tables, counted in `bytes`
    DevArray<MaterialDev> d_mats;
    std::vector<char> mat_used;           // material slots some primitive references (slot 0 of parse_obj is emissive but normally unused)
    int max_mat_index = -1;               // highest material index any primitive references: every later material set must cover it
    std::vector<Stream> streams;          // every stream and event the scene has created, destroyed with it
    std::vector<Event> events;
    // per-scene scratch, grown on demand and kept across calls
    DevArray<unsigned int> d_work;
    DevArray<unsigned long long> d_rays;
    DevArray<float4> d_tiles, d_image;
    DevArray<int> d_prim; DevArray<float> d_t;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    // wavefront integrator state (allocated on first use, grown on demand): wf_groups groups of wf_cap slots each, arrays in wf_mem
    WfGroup wf[kMaxWfGroups]{}; int wf_groups = 0, wf_cap = 0; std::vector<DevPtr> wf_mem;
    PinnedPtr h_active;                   // one word per group
    cudaEvent_t fork_event = nullptr;
    float* d_env_lum = nullptr;           // per-texel luminance as the integrator computes it (image.h:80-85), kept for the alias table
    DevArray<float2> d_alias; float alias_total = 0.0f;
    double kernel_times[4] = {};          // B200RT_FLAG_TIME_KERNELS: trace ms, shade ms, trace launches, shade launches of the last render
    WfTimeline timeline;                  // B200RT_FLAG_TIME_INLINE: per-launch events of the last wavefront frame
    bool timeline_valid = false;
    // persistent integrator state (allocated on first use)
    WfBuffers pw{}; int pw_cap = 0, pw_grid = 0; std::vector<DevPtr> pw_mem;
    // multi-GPU scenes (b200rt_scene_create_multi): this scene is rank 0; replicas[i] is rank i + 1 on another device, owned here
    std::vector<b200rt_scene*> replicas;
    DevArray<float4> d_gather;            // rank 0: world per-rank tile buffers, rank-major (the peer copies' destination)
    cudaStream_t mg_stream = nullptr;     // per device: the stream a multi-GPU frame runs on
    DevArray<unsigned char> d_rgba8;      // output stage scratch (b200rt_render_rgba8)
    // pinned staging for copies from / to pageable caller memory: two chunks, ping-pong
    PinnedPtr h_stage[2]; cudaEvent_t stage_ev[2] = { nullptr, nullptr };
    // geometry updates (b200rt_scene_update_triangles): both layouts' level lists and per-node exact boxes, made on the first update,
    // kept and counted in `bytes`; the new vertices when they have to be staged on this device
    bool refit_ready = false;
    std::vector<int> wide_level, axis_level;
    int *d_wide_idx = nullptr, *d_axis_idx = nullptr;
    float4 *d_wide_box = nullptr, *d_axis_box = nullptr;
    unsigned int* d_refit_misc = nullptr;     // [0] max |coord| bits, [1] non-finite flag, [2] quantisation overflow, [3] walk counter
    double* d_sah = nullptr;
    DevArray<float> d_vertices;

    ~b200rt_scene() { timeline.destroy(); }
};

namespace {

thread_local std::string g_error = "";

int fail(int code, const char* fmt, ...)
{
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_error = buf;
    return code;
}

#define CU(expr)                                                                                             \
    do {                                                                                                     \
        cudaError_t e__ = (expr);                                                                            \
        if (e__ != cudaSuccess) return fail(B200RT_ERR_CUDA, "%s failed: %s", #expr, cudaGetErrorString(e__)); \
    } while (0)

// Makes `device` current for the lifetime of the guard and restores the caller's device afterwards: the library must not
// change the calling thread's current device behind its back (torch and other CUDA users share the thread).
struct DeviceScope
{
    int prev = -1;
    cudaError_t err = cudaSuccess;
    explicit DeviceScope(int device)
    {
        err = cudaGetDevice(&prev);
        if (err == cudaSuccess && prev != device) err = cudaSetDevice(device);
        else if (err == cudaSuccess) prev = -1;          // nothing to restore
    }
    ~DeviceScope() { if (prev >= 0) cudaSetDevice(prev); }
    DeviceScope(const DeviceScope&) = delete;
    DeviceScope& operator=(const DeviceScope&) = delete;
};
#define ON_DEVICE(dev)                                                                                          \
    DeviceScope device_scope__(dev);                                                                             \
    if (device_scope__.err != cudaSuccess) return fail(B200RT_ERR_CUDA, "cudaSetDevice(%d) failed: %s", (dev), cudaGetErrorString(device_scope__.err))

// the library's compute has no CPU fallback: a process that sees no CUDA device gets this error from every entry point that computes
int require_device(const char* who, int* n_dev_out = nullptr)
{
    int n_dev = 0;
    if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev <= 0) return fail(B200RT_ERR_CUDA, "no CUDA device: %s has no CPU fallback", who);
    if (n_dev_out) *n_dev_out = n_dev;
    return B200RT_OK;
}

// n elements of T on the current device, owned by `owner`
template <typename T>
cudaError_t alloc_owned(std::vector<DevPtr>& owner, T** out, size_t n)
{
    void* d = nullptr;
    const cudaError_t e = cudaMalloc(&d, n * sizeof(T));
    if (e == cudaSuccess) { owner.emplace_back(d); *out = static_cast<T*>(d); }
    return e;
}

// a stream or an event on the current device, owned by the scene
int create_stream(b200rt_scene* s, cudaStream_t* out)
{
    CU(cudaStreamCreateWithFlags(out, cudaStreamNonBlocking));
    s->streams.emplace_back(*out);
    return B200RT_OK;
}

int create_event(b200rt_scene* s, cudaEvent_t* out, unsigned int flags)
{
    CU(cudaEventCreateWithFlags(out, flags));
    s->events.emplace_back(*out);
    return B200RT_OK;
}

int alloc_pinned(PinnedPtr& out, size_t bytes)
{
    void* p = nullptr;
    CU(cudaMallocHost(&p, bytes));
    out.reset(p);
    return B200RT_OK;
}

// scene data: owned by the scene and counted in its device bytes
template <typename T>
int device_alloc(b200rt_scene* s, T** out, size_t n)
{
    n = std::max<size_t>(n, 1);
    CU(alloc_owned(s->allocs, out, n));
    s->bytes += n * sizeof(T);
    return B200RT_OK;
}

template <typename T>
int upload(b200rt_scene* s, const T* host, size_t n, const T** dev_out)
{
    T* d = nullptr;
    const int rc = device_alloc(s, &d, n);
    if (rc) return rc;
    if (n) CU(cudaMemcpy(d, host, n * sizeof(T), cudaMemcpyHostToDevice));
    *dev_out = d;
    return B200RT_OK;
}

int make_params(const b200rt_scene* s, const float* camera17, int w, int h, int spp, int bounces,
                const b200rt_render_options* o, RenderParams& P)
{
    if (!s || !camera17) return fail(B200RT_ERR_ARG, "scene and camera must not be NULL");
    if (w <= 0 || h <= 0) return fail(B200RT_ERR_ARG, "bad frame size %dx%d", w, h);
    if (spp < 0 || bounces < 0) return fail(B200RT_ERR_ARG, "spp and max_bounces must be >= 0");
    b200rt_render_options d;
    b200rt_default_render_options(&d);
    if (o) d = *o;
    if (d.world <= 0) d.world = 1;
    if (d.rank < 0 || d.rank >= d.world) return fail(B200RT_ERR_ARG, "rank %d outside world %d", d.rank, d.world);
    std::memcpy(P.cam.m, camera17, 16 * sizeof(float));
    P.cam.fov_dist = camera17[16];
    P.cam.w = w; P.cam.h = h;
    P.spp = spp; P.max_bounces = bounces;
    P.rank = d.rank; P.world = d.world;
    P.tiles_x = (w + kTileDim - 1) / kTileDim;
    P.tile_skew = tile_skew();
    P.tiles_y = (h + kTileDim - 1) / kTileDim;
    P.n_rank_tiles = b200rt_tiles_for_rank(w, h, d.rank, d.world);
    P.flags = d.flags;
    P.rx0 = P.ry0 = P.rw = P.rh = 0;
    P.sample_begin = 0; P.sample_end = spp; P.acc_rng = nullptr; P.acc_sum = nullptr;
    return B200RT_OK;
}

int ensure_scratch(b200rt_scene* s, size_t tile_px, size_t image_px, size_t prim_px)
{
    CU(s->d_work.grow(1));
    CU(s->d_rays.grow(1));
    if (!s->ev1)
    {
        int rc = create_event(s, &s->ev0, cudaEventDefault);
        if (rc || (rc = create_event(s, &s->ev1, cudaEventDefault))) return rc;
    }
    CU(s->d_tiles.grow(tile_px));
    CU(s->d_image.grow(image_px));
    CU(s->d_prim.grow(prim_px));
    CU(s->d_t.grow(prim_px));
    return B200RT_OK;
}

// Runs launch() on `st`, after zeroing the scene's ray counter when count_rays, then enqueues untimed() (the copy of the result, say)
// behind it. With out != NULL, launch() is bracketed by the scene's timing events and the call returns once everything has finished,
// with the time of launch() and the ray count in *out; with out == NULL nothing is recorded and nothing waits. ensure_scratch() must
// have run.
struct LaunchResult { unsigned long long rays = 0; float ms = 0.0f; int launches = 0; };

template <typename F, typename G>
int timed_launch(b200rt_scene* s, cudaStream_t st, bool count_rays, LaunchResult* out, F launch, G untimed)
{
    if (count_rays) CU(cudaMemsetAsync(s->d_rays.get(), 0, sizeof(unsigned long long), st));
    if (out) CU(cudaEventRecord(s->ev0, st));
    int rc = launch();
    if (rc) return rc;
    if (out) CU(cudaEventRecord(s->ev1, st));
    rc = untimed();
    if (rc || !out) return rc;
    CU(cudaEventSynchronize(s->ev1));
    CU(cudaEventElapsedTime(&out->ms, s->ev0, s->ev1));
    if (count_rays) CU(cudaMemcpy(&out->rays, s->d_rays.get(), sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    return B200RT_OK;
}

template <typename F>
int timed_launch(b200rt_scene* s, cudaStream_t st, bool count_rays, LaunchResult* out, F launch)
{
    return timed_launch(s, st, count_rays, out, launch, [] { return B200RT_OK; });
}

// the stats of a call that is one timed launch sequence; kernel_ms and total_ms are both its kernel time
void launch_stats(const LaunchResult& r, b200rt_stats* stats)
{
    std::memset(stats, 0, sizeof(*stats));
    stats->kernel_ms = r.ms; stats->total_ms = r.ms; stats->rays = r.rays; stats->gpu_launches = r.launches;
}

// the integrator `opts` selects (NULL: the wavefront)
int integrator_of(const b200rt_render_options* opts, int* out)
{
    *out = opts ? opts->integrator : B200RT_INTEGRATOR_WAVEFRONT;
    if (*out < B200RT_INTEGRATOR_MEGAKERNEL || *out > B200RT_INTEGRATOR_PERSISTENT) return fail(B200RT_ERR_ARG, "unknown integrator %d", *out);
    return B200RT_OK;
}

// the scene as a launch with these flags sees it: B200RT_FLAG_ENV_ALIAS samples the env light from the alias table
int launch_scene(const b200rt_scene* s, int flags, SceneDev* out)
{
    *out = s->dev;
    if (!(flags & B200RT_FLAG_ENV_ALIAS)) return B200RT_OK;
    if (!s->d_alias.get()) return fail(B200RT_ERR_ARG, "B200RT_FLAG_ENV_ALIAS needs b200rt_scene_build_env_alias() first");
    out->use_alias = 1;
    out->cdf_total = s->alias_total;      // the normalisation the table was built with (the float running sum can be far off, see DESIGN.md)
    return B200RT_OK;
}

// pixels of the rank P names that lie inside the w x h frame
unsigned long long pixels_of_rank(const RenderParams& P, int w, int h)
{
    unsigned long long px = 0;
    for (int k = 0; k < P.n_rank_tiles; k++)
    {
        int tx, ty;
        tile_xy(P.rank + k * P.world, P.tiles_x, P.tile_skew, tx, ty);
        px += (unsigned long long)std::min(kTileDim, w - tx * kTileDim) * std::min(kTileDim, h - ty * kTileDim);
    }
    return px;
}


// ---- host <-> device copies -----------------------------------------------------------------------------------------------------
// Caller buffers may be pageable (std::vector, numpy) or page-locked (b200rt_host_alloc, cudaHostRegister). Page-locked memory
// is copied directly at the PCIe rate. Pageable memory goes through two pinned chunks owned by the scene: the DMA of one
// chunk overlaps the host memcpy of the other (a plain cudaMemcpy on pageable memory does the same inside the driver, one
// thread and smaller chunks).
constexpr size_t kStageChunk = 8u << 20;

bool host_pointer_is_pinned(const void* p)
{
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost || a.type == cudaMemoryTypeManaged;
}

void host_memcpy(void* dst, const void* src, size_t bytes)
{
    constexpr size_t kBlock = 1u << 20;
    const long long n_blocks = (long long)((bytes + kBlock - 1) / kBlock);
    if (n_blocks < 4) { std::memcpy(dst, src, bytes); return; }
#pragma omp parallel for schedule(static)
    for (long long b = 0; b < n_blocks; b++)
    {
        const size_t off = (size_t)b * kBlock;
        std::memcpy((char*)dst + off, (const char*)src + off, std::min(kBlock, bytes - off));
    }
}

int ensure_stage(b200rt_scene* s)
{
    for (int i = 0; i < 2; i++)
    {
        int rc = B200RT_OK;
        if (!s->h_stage[i] && (rc = alloc_pinned(s->h_stage[i], kStageChunk))) return rc;
        if (!s->stage_ev[i] && (rc = create_event(s, &s->stage_ev[i], cudaEventDisableTiming))) return rc;
    }
    return B200RT_OK;
}

// asynchronous with respect to the host only for pinned sources; in both cases `src` may be reused when the call returns
// only after the stream has been synchronised (pinned) or immediately (pageable: it has been copied out)
int copy_to_device(b200rt_scene* s, void* dst_dev, const void* src_host, size_t bytes, cudaStream_t st)
{
    if (!bytes) return B200RT_OK;
    if (host_pointer_is_pinned(src_host)) { CU(cudaMemcpyAsync(dst_dev, src_host, bytes, cudaMemcpyHostToDevice, st)); return B200RT_OK; }
    int rc = ensure_stage(s);
    if (rc) return rc;
    size_t off = 0;
    for (int i = 0; off < bytes; i++, off += kStageChunk)
    {
        const int b = i & 1;
        const size_t n = std::min(kStageChunk, bytes - off);
        if (i >= 2) CU(cudaEventSynchronize(s->stage_ev[b]));            // the DMA that last read this chunk has finished
        host_memcpy(s->h_stage[b].get(), (const char*)src_host + off, n);
        CU(cudaMemcpyAsync((char*)dst_dev + off, s->h_stage[b].get(), n, cudaMemcpyHostToDevice, st));
        CU(cudaEventRecord(s->stage_ev[b], st));
    }
    return B200RT_OK;
}

// blocking: returns when dst_host holds the data
int copy_to_host(b200rt_scene* s, void* dst_host, const void* src_dev, size_t bytes, cudaStream_t st)
{
    if (!bytes) { CU(cudaStreamSynchronize(st)); return B200RT_OK; }
    if (host_pointer_is_pinned(dst_host))
    {
        CU(cudaMemcpyAsync(dst_host, src_dev, bytes, cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        return B200RT_OK;
    }
    int rc = ensure_stage(s);
    if (rc) return rc;
    const size_t n_chunks = (bytes + kStageChunk - 1) / kStageChunk;
    auto issue = [&](size_t i) -> cudaError_t {
        const size_t off = i * kStageChunk, n = std::min(kStageChunk, bytes - off);
        cudaError_t e = cudaMemcpyAsync(s->h_stage[i & 1].get(), (const char*)src_dev + off, n, cudaMemcpyDeviceToHost, st);
        return e != cudaSuccess ? e : cudaEventRecord(s->stage_ev[i & 1], st);
    };
    CU(issue(0));
    if (n_chunks > 1) CU(issue(1));
    for (size_t i = 0; i < n_chunks; i++)
    {
        const size_t off = i * kStageChunk, n = std::min(kStageChunk, bytes - off);
        CU(cudaEventSynchronize(s->stage_ev[i & 1]));
        host_memcpy((char*)dst_host + off, s->h_stage[i & 1].get(), n);
        if (i + 2 < n_chunks) CU(issue(i + 2));
    }
    return B200RT_OK;
}

// the arrays of a WfBuffers of n slots, owned by `mem`
int alloc_wf_buffers(std::vector<DevPtr>& mem, WfBuffers& w, size_t n)
{
    CU(alloc_owned(mem, &w.rng, n)); CU(alloc_owned(mem, &w.sample, n)); CU(alloc_owned(mem, &w.bounce, n)); CU(alloc_owned(mem, &w.flags, n));
    CU(alloc_owned(mem, &w.final_c, n)); CU(alloc_owned(mem, &w.sample_c, n)); CU(alloc_owned(mem, &w.thr, n)); CU(alloc_owned(mem, &w.thr_next, n));
    CU(alloc_owned(mem, &w.ray_o, 5 * n)); CU(alloc_owned(mem, &w.ray_d, 5 * n)); CU(alloc_owned(mem, &w.side_w, 4 * n));
    CU(alloc_owned(mem, &w.res, 5 * n));
    CU(alloc_owned(mem, &w.queue, 5 * n)); CU(alloc_owned(mem, &w.counters, (size_t)8)); CU(alloc_owned(mem, &w.rays_total, (size_t)1));
    return B200RT_OK;
}

// tile groups (independent iteration chains on their own streams). 3 for a full 1080p frame; a rank that holds a fraction of it
// (multi-GPU) is latency-bound per pass and gains a little from a fourth chain (one rank of 8 emulated: 115.9 -> 112.2 ms)
int wavefront_group_count(const RenderParams& P)
{
    const char* e = getenv("B200RT_WF_GROUPS");          // read per frame (tools sweep it inside one process)
    const int env_n = e ? std::min(atoi(e), kMaxWfGroups) : 0;
    if (env_n >= 1) return env_n;
    return (long long)P.n_rank_tiles * kTilePixels < 700000 ? 4 : 3;
}

int ensure_wavefront(b200rt_scene* s, const RenderParams& P)
{
    const int G = wavefront_group_count(P);
    int rc = B200RT_OK;
    if (!s->fork_event)      // created last: once it exists, so do the pinned words and every group's stream and events
    {
        rc = alloc_pinned(s->h_active, kMaxWfGroups * sizeof(unsigned int));
        for (int g = 0; g < kMaxWfGroups && !rc; g++)
        {
            WfGroup& wg = s->wf[g];
            wg.host_active = static_cast<unsigned int*>(s->h_active.get()) + g;
            if (!(rc = create_stream(s, &wg.stream)) && !(rc = create_event(s, &wg.poll_event, cudaEventDisableTiming)))
                rc = create_event(s, &wg.join_event, cudaEventDisableTiming);
        }
        if (rc || (rc = create_event(s, &s->fork_event, cudaEventDisableTiming))) return rc;
    }
    // group g of rank r == rank r + g * world of a (world * G) partition
    int need[kMaxWfGroups];
    int most = 1;
    for (int g = 0; g < G; g++)
    {
        need[g] = b200rt_tiles_for_rank(P.cam.w, P.cam.h, P.rank + g * P.world, P.world * G) * kTilePixels;
        most = std::max(most, need[g]);
    }
    if (s->wf_groups != G || most > s->wf_cap)
    {
        // (re)allocate every group at the largest group's size: the buffers are then reusable for any rank/world split of
        // this frame size or smaller (the arrays are indexed k * n_slots + slot, so only the capacity matters). The old arrays are
        // freed first, so that peak device memory holds one slot state (C3's is ~780 MB), and the group count and capacity are
        // recorded only once every group's arrays exist.
        s->wf_mem.clear();
        s->wf_groups = 0; s->wf_cap = 0;
        for (WfGroup& wg : s->wf) wg.buf = WfBuffers{};
        for (int g = 0; g < G; g++)
            if ((rc = alloc_wf_buffers(s->wf_mem, s->wf[g].buf, (size_t)most))) return rc;
        s->wf_groups = G; s->wf_cap = most;
    }
    for (int g = 0; g < G; g++)
    {
        s->wf[g].buf.n_slots = need[g];
        s->wf[g].buf.tile_stride = G;
        s->wf[g].buf.tile_offset = g;
    }
    return B200RT_OK;
}

int ensure_persistent(b200rt_scene* s)
{
    const int grid = persistent_grid();
    const int n = persistent_slots(grid);
    s->pw_grid = grid;
    if (n > s->pw_cap)
    {
        // freed first and recorded once allocated, as in ensure_wavefront
        s->pw_mem.clear();
        s->pw = WfBuffers{}; s->pw_cap = 0;
        const int rc = alloc_wf_buffers(s->pw_mem, s->pw, (size_t)n);
        if (rc) return rc;
        s->pw.tile_stride = 1;
        s->pw_cap = n;
    }
    s->pw.n_slots = n;
    return B200RT_OK;
}

// runs the selected integrator for this rank's tiles on `st`; *launches receives the number of kernels launched
int run_integrator(b200rt_scene* s, const RenderParams& P, int integrator, const float4* fb_in, float4* out_tiles, cudaStream_t st, int* launches)
{
    s->kernel_times[0] = s->kernel_times[1] = s->kernel_times[2] = s->kernel_times[3] = 0.0;
    s->timeline_valid = false;
    SceneDev dev;
    int rc = launch_scene(s, P.flags, &dev);
    if (rc) return rc;
    if (integrator == B200RT_INTEGRATOR_WAVEFRONT)
    {
        if ((rc = ensure_wavefront(s, P))) return rc;
        unsigned int unfinished = 0;
        s->timeline_valid = (P.flags & B200RT_FLAG_TIME_INLINE) && !(P.flags & B200RT_FLAG_TIME_KERNELS);
        CU(run_wavefront(dev, P, s->wf, s->wf_groups, fb_in, out_tiles, st, s->fork_event, launches, s->kernel_times, &unfinished, &s->timeline));
        if (unfinished) return fail(B200RT_ERR_CUDA, "wavefront integrator: %u pixels unfinished after spp * (max_bounces + 1) iterations", unfinished);
        CU(wavefront_sum_rays(s->wf, s->wf_groups, s->d_rays.get(), st));
        *launches += 1;
        return B200RT_OK;
    }
    if (integrator == B200RT_INTEGRATOR_PERSISTENT)
    {
        if (!dev.has_wide) return fail(B200RT_ERR_ARG, "the persistent integrator traverses the 8-ary BVH (leaves of at most 3 triangles)");
        if ((rc = ensure_persistent(s))) return rc;
        CU(run_persistent(dev, P, s->pw, s->pw_grid, fb_in, out_tiles, st));
        CU(cudaMemcpyAsync(s->d_rays.get(), s->pw.rays_total, sizeof(unsigned long long), cudaMemcpyDeviceToDevice, st));
        *launches = 1;
        return B200RT_OK;
    }
    CU(launch_megakernel(dev, P, fb_in, out_tiles, s->d_work.get(), s->d_rays.get(), st));
    *launches = 1;
    return B200RT_OK;
}

// per-kernel timing fields of the stats struct (the frame must have completed)
int fill_kernel_times(b200rt_scene* s, b200rt_stats* stats)
{
    stats->trace_ms = s->kernel_times[0]; stats->shade_ms = s->kernel_times[1];
    stats->trace_launches = (int)s->kernel_times[2]; stats->shade_launches = (int)s->kernel_times[3];
    stats->trace_union_ms = 0.0; stats->tail_ms = 0.0; stats->tail_launches = 0;
    if (s->timeline_valid)
    {
        WfTimelineSummary t;
        CU(wavefront_timeline_summary(s->timeline, &t));
        stats->trace_ms = t.trace_ms; stats->shade_ms = t.shade_ms;
        stats->trace_launches = t.trace_launches; stats->shade_launches = t.shade_launches;
        stats->trace_union_ms = t.trace_union_ms;
        stats->tail_ms = t.tail_ms; stats->tail_launches = t.tail_launches;
    }
    return B200RT_OK;
}

int convert_materials(const float* materials10, int n, const std::vector<char>& used, std::vector<MaterialDev>& out, int* any_emissive)
{
    out.resize((size_t)std::max(n, 1));
    *any_emissive = 0;
    for (int i = 0; i < n; i++)
    {
        const float* m = materials10 + 10 * (size_t)i;
        MaterialDev& d = out[i];
        d.er = m[0]; d.eg = m[1]; d.eb = m[2];
        d.dr = m[4]; d.dg = m[5]; d.db = m[6];
        d.metalness = m[8]; d.roughness = m[9];
        const bool referenced = i >= (int)used.size() || used[i];
        if (referenced && (m[0] > 0.0f || m[1] > 0.0f || m[2] > 0.0f)) *any_emissive = 1;
    }
    return B200RT_OK;
}

} // namespace

extern "C" {

const char* b200rt_last_error(void) { return g_error.c_str(); }
const char* b200rt_version(void) { return "b200rt 0.1 (sm_100a)"; }

void b200rt_bvh_default_options(b200rt_bvh_options* o)
{
    if (!o) return;
    o->max_leaf_size = 3; o->sah_bins = 16; o->use_diag_slabs = 1; o->num_threads = 0;
}

void b200rt_default_render_options(b200rt_render_options* o)
{
    if (!o) return;
    o->integrator = B200RT_INTEGRATOR_WAVEFRONT; o->flags = 0; o->rank = 0; o->world = 1;
}

int b200rt_bvh_build(const float* tri_xyz9, int n_tri, const b200rt_bvh_options* opts, b200rt_bvh** out)
{
    if (!out) return fail(B200RT_ERR_ARG, "out must not be NULL");
    *out = nullptr;
    if (n_tri < 0 || (n_tri > 0 && !tri_xyz9)) return fail(B200RT_ERR_ARG, "bad triangle buffer");
    if (n_tri >= (1 << 27)) return fail(B200RT_ERR_ARG, "at most 2^27-1 triangles (leaf references pack first<<4|count)");
    b200rt_bvh_options o;
    b200rt_bvh_default_options(&o);
    if (opts) o = *opts;
    b200rt_bvh* b = new (std::nothrow) b200rt_bvh;
    if (!b) return fail(B200RT_ERR_ALLOC, "out of host memory");
    try { build_flat_bvh(tri_xyz9, n_tri, o, b->flat); }
    catch (const std::exception& e) { delete b; return fail(B200RT_ERR_ALLOC, "BVH build failed: %s", e.what()); }
    if (b->flat.info.wide_max_depth > kMaxTraversalDepth || b->flat.info.max_depth > kMaxTraversalDepth) { delete b; return fail(B200RT_ERR_ARG, "BVH depth %d exceeds the traversal stack", b->flat.info.max_depth); }
    *out = b;
    return B200RT_OK;
}

int b200rt_bvh_build_device(const float* tri_xyz9, int n_tri, int device, b200rt_bvh** out)
{
    if (!out) return fail(B200RT_ERR_ARG, "out must not be NULL");
    *out = nullptr;
    if (n_tri < 0 || (n_tri > 0 && !tri_xyz9)) return fail(B200RT_ERR_ARG, "bad triangle buffer");
    if (n_tri >= (1 << 27)) return fail(B200RT_ERR_ARG, "at most 2^27-1 triangles (leaf references pack first<<4|count)");
    if (n_tri <= kWideMaxLeaf) return b200rt_bvh_build(tri_xyz9, n_tri, nullptr, out);      // a single leaf: nothing to build in parallel
    int n_dev = 0;
    int rc = require_device("b200rt_bvh_build_device", &n_dev);
    if (rc) return rc;
    if (device < 0) CU(cudaGetDevice(&device));
    if (device >= n_dev) return fail(B200RT_ERR_ARG, "device %d of %d", device, n_dev);
    ON_DEVICE(device);
    b200rt_bvh* b = new (std::nothrow) b200rt_bvh;
    if (!b) return fail(B200RT_ERR_ALLOC, "out of host memory");
    std::string err;
    try { rc = build_flat_bvh_device(tri_xyz9, n_tri, device, b->flat, err); }
    catch (const std::exception& e) { err = e.what(); rc = 1; }
    if (rc == 2) { delete b; return b200rt_bvh_build(tri_xyz9, n_tri, nullptr, out); }     // radix tree deeper than the traversal stack: host SAH builder
    if (rc) { delete b; return fail(B200RT_ERR_CUDA, "device BVH build: %s", err.c_str()); }
    *out = b;
    return B200RT_OK;
}

int b200rt_bvh_get_info(const b200rt_bvh* bvh, b200rt_bvh_info* out)
{
    if (!bvh || !out) return fail(B200RT_ERR_ARG, "NULL argument");
    *out = bvh->flat.info;
    if (out->sah_cost == 0.0) out->sah_cost = sah_cost_of(bvh->flat);       // device-built trees: computed on request from the binary records
    return B200RT_OK;
}

int b200rt_bvh_get_arrays(const b200rt_bvh* bvh, const float** axis16, const float** diag16, const float** tris12)
{
    if (!bvh) return fail(B200RT_ERR_ARG, "NULL bvh");
    if (axis16) *axis16 = reinterpret_cast<const float*>(bvh->flat.axis.data());
    if (diag16) *diag16 = reinterpret_cast<const float*>(bvh->flat.diag.data());
    if (tris12) *tris12 = reinterpret_cast<const float*>(bvh->flat.tris.data());
    return B200RT_OK;
}

int b200rt_bvh_get_wide_nodes(const b200rt_bvh* bvh, const void** nodes80, int* n_nodes)
{
    if (!bvh || !nodes80 || !n_nodes) return fail(B200RT_ERR_ARG, "NULL argument");
    *nodes80 = bvh->flat.wide.data();
    *n_nodes = (int)bvh->flat.wide.size();
    return B200RT_OK;
}

int b200rt_bvh_check(const b200rt_bvh* bvh, const float* tri_xyz9, int n_tri)
{
    if (!bvh) return fail(B200RT_ERR_ARG, "NULL bvh");
    int r = check_flat_bvh(bvh->flat, tri_xyz9, n_tri);
    if (r) return fail(100 + r, "BVH invariant %d violated", r);
    return B200RT_OK;
}

void b200rt_bvh_destroy(b200rt_bvh* bvh) { delete bvh; }

} // extern "C"

namespace {

struct SceneArgs
{
    const float* tri_xyz9; int n_tri;
    const int* tri_material; int n_material_indices;
    const float* materials10; int n_materials;
    const int* emissive_tri; int n_emissive;
    const void* spheres20; int n_spheres;
    const float* env_rgba; int env_w, env_h; const float* env_cdf_or_null;
    int env_channels;       // 4 = Image (RGBA); 3 = stbi_loadf's RGB triplets, expanded on the device (utils.cpp:113-121)
};

int validate_scene_args(const SceneArgs& a)
{
    if (a.n_tri < 0 || (a.n_tri > 0 && !a.tri_xyz9)) return fail(B200RT_ERR_ARG, "bad triangle buffer");
    if (a.n_material_indices < a.n_tri || (a.n_material_indices > 0 && !a.tri_material)) return fail(B200RT_ERR_ARG, "need one material index per triangle");
    if (a.n_materials <= 0 || !a.materials10) return fail(B200RT_ERR_ARG, "need at least one material");
    if (a.n_emissive < 0 || (a.n_emissive > 0 && !a.emissive_tri)) return fail(B200RT_ERR_ARG, "bad emissive triangle list");
    if (a.n_spheres < 0 || (a.n_spheres > 0 && !a.spheres20)) return fail(B200RT_ERR_ARG, "bad sphere buffer");
    if (a.env_channels != 3 && a.env_channels != 4) return fail(B200RT_ERR_ARG, "env_channels must be 3 (RGB) or 4 (RGBA)");
    if (!a.env_rgba || a.env_w <= 0 || a.env_h <= 0)
        return fail(B200RT_ERR_ARG, "an environment map is required (the reference samples it unconditionally, render_kernel.cpp:114)");
    for (int i = 0; i < a.n_material_indices; i++)
        if (a.tri_material[i] < 0 || a.tri_material[i] >= a.n_materials) return fail(B200RT_ERR_ARG, "material index %d of primitive %d out of range", a.tri_material[i], i);
    for (int i = 0; i < a.n_emissive; i++)
        if (a.emissive_tri[i] < 0 || a.emissive_tri[i] >= a.n_tri) return fail(B200RT_ERR_ARG, "emissive triangle index out of range");
    return B200RT_OK;
}

// host-side products shared by every device replica of a scene (computed once)
struct SceneHostData
{
    std::vector<float4> bvh_and_tris; size_t n_wide4 = 0;
    std::vector<unsigned char> oct_lut;
    std::vector<int> slot_of_prim;
    std::vector<SphereDev> spheres;
};

void prepare_host_data(const SceneArgs& a, const FlatBVH& f, SceneHostData& h)
{
    // the 8-ary nodes and the triangle stream share one allocation (DESIGN.md §2): the triangles sit right behind the nodes
    const size_t nw = f.wide.size() * 5, nt = f.tris.size() * 3;
    h.bvh_and_tris.resize(std::max<size_t>(nw + nt, 1));
    if (nw) std::memcpy(h.bvh_and_tris.data(), f.wide.data(), nw * sizeof(float4));
    if (nt) std::memcpy(h.bvh_and_tris.data() + nw, f.tris.data(), nt * sizeof(float4));
    h.n_wide4 = nw;
    h.oct_lut.resize(8 * 256);
    for (int o = 0; o < 8; o++)
        for (int m = 0; m < 256; m++)
        {
            unsigned r = 0;
            for (int b = 0; b < 8; b++) if (m & (1 << b)) r |= 1u << (b ^ o);
            h.oct_lut[(size_t)o * 256 + m] = (unsigned char)r;
        }
    h.slot_of_prim.assign((size_t)std::max(a.n_tri, 1), 0);
    for (size_t i = 0; i < f.tris.size(); i++) h.slot_of_prim[f.tris[i].prim] = (int)i;
    h.spheres.resize((size_t)std::max(a.n_spheres, 1));
    for (int i = 0; i < a.n_spheres; i++) std::memcpy(&h.spheres[i], (const char*)a.spheres20 + 20 * (size_t)i, 20);
}

// uploads one replica of the scene to `device`
int create_on_device(const SceneArgs& a, const FlatBVH& f, const SceneHostData& h, int device, b200rt_scene** out)
{
    *out = nullptr;
    ON_DEVICE(device);
    std::unique_ptr<b200rt_scene> s(new (std::nothrow) b200rt_scene);     // frees a half-built replica on every early return
    if (!s) return fail(B200RT_ERR_ALLOC, "out of host memory");
    s->device = device;
    s->info = f.info;
    s->mat_used.assign((size_t)a.n_materials, 0);
    for (int i = 0; i < a.n_material_indices; i++) { s->mat_used[a.tri_material[i]] = 1; s->max_mat_index = std::max(s->max_mat_index, a.tri_material[i]); }
    const size_t nt = f.tris.size() * 3;
    int rc = upload(s.get(), h.bvh_and_tris.data(), h.n_wide4 + nt, &s->dev.wide);
    if (rc) return rc;
    s->dev.tris = s->dev.wide + h.n_wide4;
    s->dev.has_wide = f.wide.empty() ? 0 : 1;
    s->dev.qmagic = 0x43000000u;
    if ((rc = upload(s.get(), h.oct_lut.data(), h.oct_lut.size(), &s->dev.oct_lut))) return rc;
    if ((rc = upload(s.get(), reinterpret_cast<const float4*>(f.axis.data()), f.axis.size() * 4, &s->dev.axis))) return rc;
    if ((rc = upload(s.get(), reinterpret_cast<const float4*>(f.diag.data()), f.diag.size() * 4, &s->dev.diag))) return rc;
    if ((rc = upload(s.get(), h.slot_of_prim.data(), (size_t)a.n_tri, &s->dev.slot_of_prim))) return rc;
    if ((rc = upload(s.get(), a.tri_material, (size_t)a.n_material_indices, &s->dev.mat_idx))) return rc;
    if ((rc = upload(s.get(), a.emissive_tri, (size_t)a.n_emissive, &s->dev.emissive))) return rc;
    if ((rc = upload(s.get(), h.spheres.data(), (size_t)a.n_spheres, &s->dev.spheres))) return rc;
    const size_t n_texels = (size_t)a.env_w * a.env_h;
    if (a.env_channels == 3)
    {
        float4* d_env = nullptr;
        if ((rc = device_alloc(s.get(), &d_env, n_texels))) return rc;
        DevArray<float> rgb;
        cudaError_t ce = rgb.grow(n_texels * 3);
        if (ce == cudaSuccess) ce = cudaMemcpy(rgb.get(), a.env_rgba, n_texels * 3 * sizeof(float), cudaMemcpyHostToDevice);
        if (ce == cudaSuccess) ce = launch_env_expand_rgb(rgb.get(), n_texels, d_env, 0);
        if (ce == cudaSuccess) ce = cudaDeviceSynchronize();
        if (ce != cudaSuccess) return fail(B200RT_ERR_CUDA, "env RGB -> RGBA: %s", cudaGetErrorString(ce));
        s->dev.env = d_env;
    }
    else if ((rc = upload(s.get(), reinterpret_cast<const float4*>(a.env_rgba), n_texels, &s->dev.env))) return rc;
    s->dev.n_tri = a.n_tri; s->dev.n_emissive = a.n_emissive; s->dev.n_spheres = a.n_spheres;
    s->dev.env_w = a.env_w; s->dev.env_h = a.env_h;
    s->dev.has_diag = f.info.has_diag_slabs;
    // env tables (K5, env_tables.cu): per-texel luminance, the running-sum CDF in the reference's serial float order
    // (Utils::compute_env_map_cdf, utils.cpp:126-142) unless the caller brings its own, and the last-column copy the row search probes
    float* d_lum = nullptr; float* d_cdf = nullptr; float* d_row = nullptr;
    if ((rc = device_alloc(s.get(), &d_lum, n_texels)) || (rc = device_alloc(s.get(), &d_cdf, n_texels)) || (rc = device_alloc(s.get(), &d_row, (size_t)a.env_h))) return rc;
    cudaError_t ce = launch_env_luminance(s->dev.env, n_texels, d_lum, 0);
    if (ce == cudaSuccess)
    {
        if (a.env_cdf_or_null) ce = cudaMemcpy(d_cdf, a.env_cdf_or_null, n_texels * sizeof(float), cudaMemcpyHostToDevice);
        else ce = launch_env_cdf_serial(d_lum, n_texels, d_cdf, 0);
    }
    if (ce == cudaSuccess) ce = launch_env_row_cdf(d_cdf, a.env_w, a.env_h, d_row, 0);
    if (ce == cudaSuccess) ce = cudaMemcpy(&s->dev.cdf_total, d_cdf + n_texels - 1, sizeof(float), cudaMemcpyDeviceToHost);
    if (ce != cudaSuccess) return fail(B200RT_ERR_CUDA, "env tables: %s", cudaGetErrorString(ce));
    s->dev.cdf = d_cdf; s->dev.row_cdf = d_row; s->d_env_lum = d_lum;
    // guide table of the CDF search (bit-identical texel choice, ~2 probes instead of log2(W) + log2(H)); B200RT_CDF_GUIDE=0 turns it off
    static const int guide_buckets = []() { const char* e = getenv("B200RT_CDF_GUIDE"); int v = e ? atoi(e) : 65536; return v < 0 ? 0 : v; }();
    if (guide_buckets > 0 && n_texels >= 64)
    {
        unsigned int* d_guide = nullptr;
        if ((rc = device_alloc(s.get(), &d_guide, (size_t)guide_buckets + 2))) return rc;
        float scale = 0.0f; int built = 0;
        ce = build_env_cdf_guide(d_cdf, n_texels, s->dev.cdf_total, guide_buckets, d_guide, &scale, &built, 0);
        if (ce != cudaSuccess) return fail(B200RT_ERR_CUDA, "env CDF guide: %s", cudaGetErrorString(ce));
        if (built) { s->dev.cdf_guide = d_guide; s->dev.cdf_guide_scale = scale; s->dev.cdf_guide_n = guide_buckets; }
    }
    if ((rc = b200rt_scene_set_materials(s.get(), a.materials10, a.n_materials))) return rc;
    *out = s.release();
    return B200RT_OK;
}

int create_scene(const SceneArgs& a, const b200rt_bvh* bvh_or_null, const int* devices, int n_devices, b200rt_scene** out)
{
    if (!out) return fail(B200RT_ERR_ARG, "out must not be NULL");
    *out = nullptr;
    int rc = validate_scene_args(a);
    if (rc) return rc;
    int n_dev = 0;
    if ((rc = require_device("b200rt", &n_dev))) return rc;
    if (n_devices <= 0 || n_devices > 64) return fail(B200RT_ERR_ARG, "bad device count %d", n_devices);
    std::vector<int> devs((size_t)n_devices);
    for (int i = 0; i < n_devices; i++)
    {
        int d = devices ? devices[i] : -1;
        if (d < 0) { if (n_devices > 1) d = i; else CU(cudaGetDevice(&d)); }
        if (d >= n_dev) return fail(B200RT_ERR_ARG, "device %d of %d", d, n_dev);
        devs[i] = d;
    }

    b200rt_bvh* own = nullptr;
    const b200rt_bvh* bvh = bvh_or_null;
    if (!bvh)
    {
        // above ~5 M triangles the host SAH build dominates the whole job (12.5 s at 20 M, DESIGN.md): build on the GPU instead
        static const int device_build_threshold = []() { const char* e = getenv("B200RT_DEVICE_BUILD_MIN_TRIS"); return e ? atoi(e) : 5000000; }();
        rc = a.n_tri >= device_build_threshold ? b200rt_bvh_build_device(a.tri_xyz9, a.n_tri, devs[0], &own) : b200rt_bvh_build(a.tri_xyz9, a.n_tri, nullptr, &own);
        if (rc) return rc;
        bvh = own;
    }
    if (bvh->flat.info.n_triangles != a.n_tri) { delete own; return fail(B200RT_ERR_ARG, "BVH was built for %d triangles, scene has %d", bvh->flat.info.n_triangles, a.n_tri); }

    SceneHostData h;
    prepare_host_data(a, bvh->flat, h);
    b200rt_scene* first = nullptr;
    rc = create_on_device(a, bvh->flat, h, devs[0], &first);
    for (int i = 1; i < n_devices && !rc; i++)
    {
        b200rt_scene* r = nullptr;
        rc = create_on_device(a, bvh->flat, h, devs[i], &r);
        if (!rc) first->replicas.push_back(r);
    }
    delete own;
    if (rc) { if (first) b200rt_scene_destroy(first); return rc; }
    if (n_devices > 1)
    {
        // peer access towards rank 0's device: the per-rank tile buffers are copied GPU to GPU (NVLink) at the end of a frame
        for (b200rt_scene* r : first->replicas)
        {
            DeviceScope scope(r->device);
            int can = 0;
            if (cudaDeviceCanAccessPeer(&can, r->device, first->device) == cudaSuccess && can)
            {
                const cudaError_t pe = cudaDeviceEnablePeerAccess(first->device, 0);
                if (pe != cudaSuccess) cudaGetLastError();      // already enabled (or unsupported: the copy is then staged by the driver)
            }
        }
    }
    *out = first;
    return B200RT_OK;
}

} // namespace

extern "C" {

int b200rt_scene_create(const float* tri_xyz9, int n_tri, const int* tri_material, int n_material_indices,
                        const float* materials10, int n_materials, const int* emissive_tri, int n_emissive,
                        const void* spheres20, int n_spheres,
                        const float* env_rgba, int env_w, int env_h, const float* env_cdf_or_null,
                        const b200rt_bvh* bvh_or_null, int device, b200rt_scene** out)
{
    const SceneArgs a = { tri_xyz9, n_tri, tri_material, n_material_indices, materials10, n_materials, emissive_tri, n_emissive,
                          spheres20, n_spheres, env_rgba, env_w, env_h, env_cdf_or_null, 4 };
    return create_scene(a, bvh_or_null, &device, 1, out);
}

int b200rt_scene_create_multi(const float* tri_xyz9, int n_tri, const int* tri_material, int n_material_indices,
                              const float* materials10, int n_materials, const int* emissive_tri, int n_emissive,
                              const void* spheres20, int n_spheres,
                              const float* env_pixels, int env_channels, int env_w, int env_h, const float* env_cdf_or_null,
                              const b200rt_bvh* bvh_or_null, const int* devices_or_null, int n_devices, b200rt_scene** out)
{
    const SceneArgs a = { tri_xyz9, n_tri, tri_material, n_material_indices, materials10, n_materials, emissive_tri, n_emissive,
                          spheres20, n_spheres, env_pixels, env_w, env_h, env_cdf_or_null, env_channels };
    return create_scene(a, bvh_or_null, devices_or_null, n_devices, out);
}

int b200rt_scene_device_count(const b200rt_scene* s) { return s ? 1 + (int)s->replicas.size() : 0; }

// Vose's alias method in double over per-texel luminances: texel i is accepted with probability prob[i], otherwise alias[i] is taken
static int build_alias_table(const float* lum, size_t n, std::vector<float>& prob, std::vector<int>& alias_out, double* total_out)
{
    double total = 0.0;
    for (size_t i = 0; i < n; i++) total += lum[i] > 0.0f ? (double)lum[i] : 0.0;
    if (!(total > 0.0)) return fail(B200RT_ERR_ARG, "environment map has no luminance to sample");
    std::vector<double> q(n);
    std::vector<unsigned int> alias(n), small, large;
    small.reserve(n); large.reserve(n);
    for (size_t i = 0; i < n; i++)
    {
        q[i] = (lum[i] > 0.0f ? (double)lum[i] : 0.0) / total * (double)n;
        alias[i] = (unsigned int)i;
        (q[i] < 1.0 ? small : large).push_back((unsigned int)i);
    }
    while (!small.empty() && !large.empty())
    {
        const unsigned int lo = small.back(), hi = large.back();
        small.pop_back();
        alias[lo] = hi;
        q[hi] = (q[hi] + q[lo]) - 1.0;
        if (q[hi] < 1.0) { large.pop_back(); small.push_back(hi); }
    }
    for (unsigned int i : large) q[i] = 1.0;
    for (unsigned int i : small) q[i] = 1.0;          // numerical leftovers
    prob.resize(n); alias_out.resize(n);
    for (size_t i = 0; i < n; i++) { prob[i] = (float)q[i]; alias_out[i] = (int)alias[i]; }
    *total_out = total;
    return B200RT_OK;
}

int b200rt_env_alias_table(const float* env_rgba, int env_w, int env_h, float* prob_out, int* alias_out, double* total_out)
{
    if (!env_rgba || env_w <= 0 || env_h <= 0 || !prob_out || !alias_out) return fail(B200RT_ERR_ARG, "bad alias table arguments");
    const size_t n = (size_t)env_w * env_h;
    std::vector<float> lum(n);
    for (size_t i = 0; i < n; i++)
    {
        const float* p = env_rgba + 4 * i;
        lum[i] = (float)(0.3086 * p[0] + 0.6094 * p[1] + 0.0820 * p[2]);      // Image::luminance_of_pixel, image.h:80-85
    }
    std::vector<float> prob; std::vector<int> alias; double total = 0.0;
    int rc = build_alias_table(lum.data(), n, prob, alias, &total);
    if (rc) return rc;
    std::memcpy(prob_out, prob.data(), n * sizeof(float));
    std::memcpy(alias_out, alias.data(), n * sizeof(int));
    if (total_out) *total_out = total;
    return B200RT_OK;
}

int b200rt_scene_build_env_alias(b200rt_scene* s)
{
    if (!s) return fail(B200RT_ERR_ARG, "NULL scene");
    for (b200rt_scene* r : s->replicas) { const int rc = b200rt_scene_build_env_alias(r); if (rc) return rc; }
    if (s->d_alias.get()) return B200RT_OK;
    ON_DEVICE(s->device);
    const size_t n = (size_t)s->dev.env_w * s->dev.env_h;
    if (!n || !s->d_env_lum) return fail(B200RT_ERR_ARG, "scene has no environment map");
    DevArray<float2> d;
    CU(d.grow(n));
    double total = 0.0;
    const cudaError_t ce = build_env_alias_device(s->d_env_lum, n, d.get(), &total, 0);
    if (ce == cudaErrorInvalidValue) { cudaGetLastError(); return fail(B200RT_ERR_ARG, "environment map has no luminance to sample"); }
    if (ce != cudaSuccess) return fail(B200RT_ERR_CUDA, "alias table build failed: %s", cudaGetErrorString(ce));
    // published together, only after the build succeeded
    s->dev.env_alias = d.get();
    s->d_alias = std::move(d);
    s->bytes += n * sizeof(float2);
    s->alias_total = (float)total;
    return B200RT_OK;
}

int b200rt_scene_get_env_alias(b200rt_scene* s, float* prob_out, int* alias_out, double* total_out)
{
    if (!s || !prob_out || !alias_out) return fail(B200RT_ERR_ARG, "NULL argument");
    if (!s->d_alias.get()) return fail(B200RT_ERR_ARG, "no alias table: call b200rt_scene_build_env_alias() first");
    ON_DEVICE(s->device);
    const size_t n = (size_t)s->dev.env_w * s->dev.env_h;
    std::vector<float2> t(n);
    CU(cudaMemcpy(t.data(), s->d_alias.get(), n * sizeof(float2), cudaMemcpyDeviceToHost));
    for (size_t i = 0; i < n; i++) { prob_out[i] = t[i].x; std::memcpy(&alias_out[i], &t[i].y, sizeof(int)); }
    if (total_out) *total_out = (double)s->alias_total;
    return B200RT_OK;
}

int b200rt_scene_get_env_cdf(b200rt_scene* s, float* cdf_out)
{
    if (!s || !cdf_out) return fail(B200RT_ERR_ARG, "NULL argument");
    ON_DEVICE(s->device);
    CU(cudaMemcpy(cdf_out, s->dev.cdf, (size_t)s->dev.env_w * s->dev.env_h * sizeof(float), cudaMemcpyDeviceToHost));
    return B200RT_OK;
}

int b200rt_scene_set_materials(b200rt_scene* s, const float* materials10, int n_materials)
{
    if (!s || !materials10 || n_materials <= 0) return fail(B200RT_ERR_ARG, "bad materials");
    if (n_materials <= s->max_mat_index)
        return fail(B200RT_ERR_ARG, "%d materials, but the scene's primitives reference material index %d", n_materials, s->max_mat_index);
    for (b200rt_scene* r : s->replicas) { const int rc = b200rt_scene_set_materials(r, materials10, n_materials); if (rc) return rc; }
    ON_DEVICE(s->device);
    std::vector<MaterialDev> mats;
    int any = 0;
    convert_materials(materials10, n_materials, s->mat_used, mats, &any);
    if ((size_t)n_materials > s->d_mats.cap)
    {
        // allocated before the old table is released: if this fails, the scene keeps rendering with its current materials
        DevArray<MaterialDev> bigger;
        CU(bigger.grow((size_t)n_materials));
        s->dev.mats = bigger.get();
        s->d_mats = std::move(bigger);
    }
    CU(cudaMemcpy(s->d_mats.get(), mats.data(), sizeof(MaterialDev) * (size_t)n_materials, cudaMemcpyHostToDevice));
    s->dev.n_mats = n_materials;
    s->dev.any_emissive_material = any;
    return B200RT_OK;
}

void b200rt_scene_destroy(b200rt_scene* s)
{
    if (!s) return;
    for (b200rt_scene* r : s->replicas) b200rt_scene_destroy(r);
    s->replicas.clear();
    DeviceScope scope(s->device);
    delete s;
}

int b200rt_scene_get_bvh_info(const b200rt_scene* s, b200rt_bvh_info* out)
{
    if (!s || !out) return fail(B200RT_ERR_ARG, "NULL argument");
    *out = s->info;
    return B200RT_OK;
}

size_t b200rt_scene_device_bytes(const b200rt_scene* s)
{
    if (!s) return 0;
    size_t b = s->bytes;
    for (const b200rt_scene* r : s->replicas) b += r->bytes;
    return b;
}

int b200rt_tiles_for_rank(int width, int height, int rank, int world)
{
    if (width <= 0 || height <= 0 || world <= 0 || rank < 0 || rank >= world) return 0;
    const int n = ((width + kTileDim - 1) / kTileDim) * ((height + kTileDim - 1) / kTileDim);
    return (n - rank + world - 1) / world;       // tiles rank, rank + world, ... < n
}

int b200rt_render_tiles_device(b200rt_scene* s, const float* camera17, int w, int h, int spp, int bounces,
                               void* dev_tiles, const b200rt_render_options* opts, void* cuda_stream, b200rt_stats* stats)
{
    RenderParams P;
    int rc = make_params(s, camera17, w, h, spp, bounces, opts, P);
    if (rc) return rc;
    if (!dev_tiles) return fail(B200RT_ERR_ARG, "dev_tiles must not be NULL");
    int integrator = 0;
    if ((rc = integrator_of(opts, &integrator))) return rc;
    ON_DEVICE(s->device);
    if ((rc = ensure_scratch(s, 0, 0, 0))) return rc;
    cudaStream_t st = (cudaStream_t)cuda_stream;
    LaunchResult r;
    rc = timed_launch(s, st, true, stats ? &r : nullptr, [&] { return run_integrator(s, P, integrator, nullptr, (float4*)dev_tiles, st, &r.launches); });
    if (rc || !stats) return rc;
    launch_stats(r, stats);
    stats->samples = pixels_of_rank(P, w, h) * (unsigned long long)spp;
    return fill_kernel_times(s, stats);
}

int b200rt_untile_device(b200rt_scene* s, const void* dev_gathered, int tiles_per_rank_padded, int world, int w, int h,
                         void* dev_image, void* cuda_stream)
{
    if (!s || !dev_gathered || !dev_image || world <= 0 || w <= 0 || h <= 0) return fail(B200RT_ERR_ARG, "bad untile arguments");
    if (tiles_per_rank_padded < b200rt_tiles_for_rank(w, h, 0, world)) return fail(B200RT_ERR_ARG, "tiles_per_rank_padded too small");
    ON_DEVICE(s->device);
    CU(launch_untile((const float4*)dev_gathered, tiles_per_rank_padded, world, -1, w, h, (float4*)dev_image, (cudaStream_t)cuda_stream));
    return B200RT_OK;
}

} // extern "C"

namespace {

// the stream a rank of a multi-GPU frame or accumulation runs on, created on the rank's device on first use
int ensure_rank_stream(b200rt_scene* r)
{
    if (r->mg_stream) return B200RT_OK;
    ON_DEVICE(r->device);
    return create_stream(r, &r->mg_stream);
}

// One rank's share of a frame or of an accumulation chunk: the integrator over the tiles P names, into `tiles`, on stream `st` of
// the rank's device. Returns when it has finished, with its kernel time and ray count in *out.
int integrate_rank(b200rt_scene* r, const RenderParams& P, int integrator, float4* tiles, cudaStream_t st, LaunchResult* out)
{
    ON_DEVICE(r->device);
    const int rc = ensure_scratch(r, 0, 0, 0);
    if (rc) return rc;
    return timed_launch(r, st, true, out, [&] { return run_integrator(r, P, integrator, nullptr, tiles, st, &out->launches); });
}

// The output stage of a frame that is in s->d_image (w x h): the float image into fb_out, or its RGBA8 quantisation, made on the
// device, into rgba8_out (exactly one is non-NULL). Returns when the caller's buffer holds it.
int output_stage(b200rt_scene* s, int w, int h, float* fb_out, unsigned char* rgba8_out, int flip_y, cudaStream_t st)
{
    const size_t image_px = (size_t)w * h;
    if (!rgba8_out) return copy_to_host(s, fb_out, s->d_image.get(), image_px * sizeof(float4), st);
    CU(s->d_rgba8.grow(image_px * 4));
    CU(launch_quantise_rgba8(s->d_image.get(), w, h, flip_y, s->d_rgba8.get(), st));
    return copy_to_host(s, rgba8_out, s->d_rgba8.get(), image_px * 4, st);
}

// rank `rank`'s n_tiles tiles into its slice of rank 0's gather buffer: ONE device-to-device copy on the rank's stream (NVLink peer
// copy; a plain copy when the rank shares rank 0's device). Returns when the copy has finished.
int gather_rank(b200rt_scene* r, b200rt_scene* root, const float4* tiles, int rank, int n_tiles, size_t tiles_padded)
{
    if (n_tiles <= 0) return B200RT_OK;
    int rc = ensure_rank_stream(r);
    if (rc) return rc;
    ON_DEVICE(r->device);
    float4* dst = root->d_gather.get() + (size_t)rank * tiles_padded * kTilePixels;
    CU(cudaMemcpyPeerAsync(dst, root->device, tiles, r->device, (size_t)n_tiles * kTilePixels * sizeof(float4), r->mg_stream));
    CU(cudaStreamSynchronize(r->mg_stream));
    return B200RT_OK;
}

// Runs rank_body(d) for every rank d < n_dev: rank 0 on the calling thread, every other rank on a host thread of its own, so that
// each device launches and waits on its own. A failure is reported as the lowest failing rank's: "device rank d: ...".
template <typename F>
int run_ranks(int n_dev, F rank_body)
{
    std::vector<int> rc((size_t)n_dev, B200RT_OK);
    std::vector<std::string> err((size_t)n_dev);
    auto run = [&](int d) { rc[(size_t)d] = rank_body(d); if (rc[(size_t)d]) err[(size_t)d] = g_error; };
    std::vector<std::thread> threads;
    for (int d = 1; d < n_dev; d++) threads.emplace_back(run, d);
    run(0);
    for (std::thread& t : threads) t.join();
    for (int d = 0; d < n_dev; d++)
        if (rc[(size_t)d]) { g_error = "device rank " + std::to_string(d) + ": " + err[(size_t)d]; return rc[(size_t)d]; }
    return B200RT_OK;
}

// The refit state of one replica: level lists by a breadth-first walk of the resident records (which it only reads) and the per-node
// exact-box arrays. Made once; a failure leaves the scene as it was, and the next update tries again.
int ensure_refit(b200rt_scene* r)
{
    if (r->refit_ready) return B200RT_OK;
    ON_DEVICE(r->device);
    const size_t n_wide = (size_t)r->info.n_wide_nodes, n_axis = (size_t)r->info.n_inner_nodes;
    int rc = B200RT_OK;
    if (!r->d_refit_misc && (rc = device_alloc(r, &r->d_refit_misc, 4))) return rc;
    if (!r->d_sah && (rc = device_alloc(r, &r->d_sah, refit_sah_scratch_doubles()))) return rc;
    if (!r->d_wide_idx && (rc = device_alloc(r, &r->d_wide_idx, n_wide))) return rc;
    if (!r->d_axis_idx && (rc = device_alloc(r, &r->d_axis_idx, n_axis))) return rc;
    if (!r->d_wide_box && (rc = device_alloc(r, &r->d_wide_box, 2 * n_wide))) return rc;
    if (!r->d_axis_box && (rc = device_alloc(r, &r->d_axis_box, 4 * n_axis))) return rc;
    const cudaError_t e = refit_levels(reinterpret_cast<const WideNode*>(r->dev.wide), (int)n_wide, reinterpret_cast<const AxisNode*>(r->dev.axis),
                                       (int)n_axis, r->d_wide_idx, r->d_axis_idx, reinterpret_cast<int*>(r->d_refit_misc + 3),
                                       r->wide_level, r->axis_level, 0);
    if (e == cudaErrorInvalidValue) return fail(B200RT_ERR_ARG, "the scene's BVH records do not form one tree rooted at record 0");
    if (e != cudaSuccess) return fail(B200RT_ERR_CUDA, "BVH level lists: %s", cudaGetErrorString(e));
    r->refit_ready = true;
    return B200RT_OK;
}

// Refits replica r to the new vertices `v` (on r's device) on stream st: triangle stream, both layouts level by level, the SAH cost.
// Returns when it has finished, with the kernel time and the launch count in *out.
int refit_rank(b200rt_scene* r, const float* v, float abs_pad, cudaStream_t st, LaunchResult* out)
{
    ON_DEVICE(r->device);
    int* overflow = reinterpret_cast<int*>(r->d_refit_misc + 2);
    CU(cudaMemsetAsync(overflow, 0, sizeof(int), st));
    RefitArgs A;
    A.tri9 = v;
    A.tris = const_cast<float4*>(r->dev.tris);
    A.wide = reinterpret_cast<WideNode*>(const_cast<float4*>(r->dev.wide));
    A.axis = reinterpret_cast<AxisNode*>(const_cast<float4*>(r->dev.axis));
    A.diag = r->dev.has_diag ? reinterpret_cast<DiagNode*>(const_cast<float4*>(r->dev.diag)) : nullptr;
    A.wide_idx = r->d_wide_idx; A.axis_idx = r->d_axis_idx;
    A.wide_level = &r->wide_level; A.axis_level = &r->axis_level;
    A.wide_box = r->d_wide_box; A.axis_box = r->d_axis_box;
    A.n_tri = r->dev.n_tri; A.n_axis = r->info.n_inner_nodes;
    A.abs_pad = abs_pad;
    A.overflow = overflow;
    A.sah = r->d_sah;
    int flag = 0;
    double sah = 0.0;
    const int rc = timed_launch(r, st, false, out, [&] { CU(refit_tree(A, st, &out->launches)); return B200RT_OK; }, [&] {
        CU(cudaMemcpyAsync(&flag, overflow, sizeof(int), cudaMemcpyDeviceToHost, st));
        CU(cudaMemcpyAsync(&sah, r->d_sah + refit_sah_scratch_doubles() - 1, sizeof(double), cudaMemcpyDeviceToHost, st));
        return B200RT_OK;
    });
    if (rc) return rc;
    CU(cudaStreamSynchronize(st));
    if (flag) return fail(B200RT_ERR_CUDA, "wide BVH quantisation overflow in the refit");
    r->info.sah_cost = sah;
    return B200RT_OK;
}

// b200rt_scene_update_triangles[_device]: new vertices for every replica of the scene. src is host memory, or (src_on_device) device
// memory of the scene's first device that the caller's stream `caller_st` produces.
int update_triangles(b200rt_scene* s, const void* src, bool src_on_device, int n_tri, cudaStream_t caller_st, b200rt_stats* stats)
{
    if (!s || !src) return fail(B200RT_ERR_ARG, "scene and triangle buffer must not be NULL");
    if (n_tri != s->dev.n_tri) return fail(B200RT_ERR_ARG, "%d triangles, but the scene has %d (an update keeps the topology)", n_tri, s->dev.n_tri);
    if (stats) std::memset(stats, 0, sizeof(*stats));
    if (n_tri == 0) return B200RT_OK;
    int rc = require_device("b200rt_scene_update_triangles");
    if (rc) return rc;
    const auto t0 = std::chrono::high_resolution_clock::now();
    if (src_on_device)
    {
        cudaPointerAttributes pa;
        if (cudaPointerGetAttributes(&pa, src) != cudaSuccess) { cudaGetLastError(); pa.type = cudaMemoryTypeUnregistered; }
        if (!((pa.type == cudaMemoryTypeDevice && pa.device == s->device) || pa.type == cudaMemoryTypeManaged))
            return fail(B200RT_ERR_ARG, "dev_tri_xyz9 must be device memory of the scene's first device (%d)", s->device);
    }
    std::vector<b200rt_scene*> ranks(1, s);
    ranks.insert(ranks.end(), s->replicas.begin(), s->replicas.end());
    const int n_dev = (int)ranks.size();
    const size_t bytes = 9 * (size_t)n_tri * sizeof(float);
    // 1. every replica's state and buffers: nothing resident is written yet
    for (int d = 0; d < n_dev; d++)
    {
        b200rt_scene* r = ranks[(size_t)d];
        if ((rc = ensure_refit(r))) return rc;
        ON_DEVICE(r->device);
        if ((rc = ensure_scratch(r, 0, 0, 0))) return rc;
        if (d > 0 && (rc = ensure_rank_stream(r))) return rc;
        if ((d > 0 || !src_on_device) && r->d_vertices.cap < 9 * (size_t)n_tri) CU(r->d_vertices.grow(9 * (size_t)n_tri));
    }
    // 2. the first device: the input there, then the extent pass; a non-finite coordinate refuses the update
    ON_DEVICE(s->device);
    const cudaStream_t st0 = src_on_device ? caller_st : 0;
    const float* v0 = src_on_device ? static_cast<const float*>(src) : s->d_vertices.get();
    if (!src_on_device && (rc = copy_to_device(s, s->d_vertices.get(), src, bytes, st0))) return rc;
    LaunchResult extent;
    extent.launches = 1;
    unsigned int misc[2] = { 0, 0 };
    rc = timed_launch(s, st0, false, &extent, [&] { CU(refit_extent(v0, n_tri, s->d_refit_misc, st0)); return B200RT_OK; },
                      [&] { CU(cudaMemcpyAsync(misc, s->d_refit_misc, sizeof(misc), cudaMemcpyDeviceToHost, st0)); return B200RT_OK; });
    if (rc) return rc;
    CU(cudaStreamSynchronize(st0));
    if (misc[1]) return fail(B200RT_ERR_ARG, "a vertex coordinate is NaN or infinite: no refitted box can bound it");
    float scene_abs;
    std::memcpy(&scene_abs, &misc[0], sizeof(float));
    const float abs_pad = 2e-6f * scene_abs + 1e-30f;          // as both builders derive it
    // 3. every replica refits on its own device, from one host thread each; the others receive the vertices first
    std::vector<LaunchResult> res((size_t)n_dev);
    rc = run_ranks(n_dev, [&](int d) -> int {
        if (d == 0) return refit_rank(s, v0, abs_pad, st0, &res[0]);
        b200rt_scene* r = ranks[(size_t)d];
        ON_DEVICE(r->device);
        if (src_on_device) CU(cudaMemcpyPeerAsync(r->d_vertices.get(), r->device, src, s->device, bytes, r->mg_stream));
        else
        {
            const int rc_c = copy_to_device(r, r->d_vertices.get(), src, bytes, r->mg_stream);
            if (rc_c) return rc_c;
        }
        return refit_rank(r, r->d_vertices.get(), abs_pad, r->mg_stream, &res[(size_t)d]);
    });
    if (rc) return rc;
    if (stats)
    {
        float ms = 0.0f;
        stats->gpu_launches = extent.launches;
        for (const LaunchResult& r : res) { ms = std::max(ms, r.ms); stats->gpu_launches += r.launches; }
        stats->kernel_ms = extent.ms + ms;
        stats->h2d_bytes = src_on_device ? 0 : bytes * (unsigned long long)n_dev;
        stats->total_ms = std::chrono::duration<double, std::milli>(std::chrono::high_resolution_clock::now() - t0).count();
    }
    return B200RT_OK;
}

// One rank of a multi-GPU frame: render this device's interleaved tiles as mean radiance (B200RT_FLAG_LINEAR_TILES) and push them
// into rank 0's gather buffer. Rank 0 renders straight into its slice of the gather buffer.
int render_rank(b200rt_scene* r, b200rt_scene* root, const RenderParams& P, int integrator, size_t tiles_padded, LaunchResult* out)
{
    ON_DEVICE(r->device);
    int rc = ensure_scratch(r, r == root ? 0 : tiles_padded * kTilePixels, 0, 0);
    if (rc) return rc;
    if ((rc = ensure_rank_stream(r))) return rc;
    if (r == root) return integrate_rank(r, P, integrator, root->d_gather.get() + (size_t)P.rank * tiles_padded * kTilePixels, r->mg_stream, out);
    if ((rc = integrate_rank(r, P, integrator, r->d_tiles.get(), r->mg_stream, out))) return rc;
    return gather_rank(r, root, r->d_tiles.get(), P.rank, P.n_rank_tiles, tiles_padded);
}

// The whole frame: framebuffer in (or Color::Black()), integrator on one or several devices, un-tile, optional RGBA8 output
// stage, result out. fb_out / rgba8_out: exactly one is non-NULL.
int render_frame(b200rt_scene* s, const float* camera17, int w, int h, int spp, int bounces, const float* fb_in, float* fb_out,
                 unsigned char* rgba8_out, int flip_y, const b200rt_render_options* opts, b200rt_stats* stats)
{
    RenderParams P;
    int rc = make_params(s, camera17, w, h, spp, bounces, opts, P);
    if (rc) return rc;
    int integrator = 0;
    if ((rc = integrator_of(opts, &integrator))) return rc;
    if (P.flags & B200RT_FLAG_LINEAR_TILES) return fail(B200RT_ERR_ARG, "B200RT_FLAG_LINEAR_TILES is for b200rt_render_tiles_device");
    const int n_dev = 1 + (int)s->replicas.size();
    if (n_dev > 1 && P.world != 1) return fail(B200RT_ERR_ARG, "a multi-GPU scene partitions the frame itself: rank/world must stay 0/1");
    auto t0 = std::chrono::high_resolution_clock::now();
    ON_DEVICE(s->device);
    const size_t image_px = (size_t)w * h;
    if ((rc = ensure_scratch(s, (size_t)std::max(P.n_rank_tiles, 1) * kTilePixels, image_px, 0))) return rc;
    cudaStream_t st = 0;
    unsigned long long h2d = 17 * sizeof(float);
    LaunchResult frame;            // kernel_ms: the slowest rank's
    const bool fb_zero = !fb_in || (P.flags & B200RT_FLAG_FB_IS_ZERO);
    float4* image = s->d_image.get();

    if (n_dev == 1)
    {
        // single device: the integrator tone-maps each finished pixel against the incoming framebuffer itself
        const bool upload_fb = !fb_zero || (P.world > 1 && fb_in);
        if (upload_fb) { if ((rc = copy_to_device(s, image, fb_in, image_px * sizeof(float4), st))) return rc; h2d += image_px * sizeof(float4); }
        else if (P.world > 1) CU(launch_fill_f4(image, image_px, make_float4(0.0f, 0.0f, 0.0f, 1.0f), st));
        auto integrate_untile = [&] {
            const int rc_i = run_integrator(s, P, integrator, fb_zero ? nullptr : image, s->d_tiles.get(), st, &frame.launches);
            if (rc_i) return rc_i;
            CU(launch_untile(s->d_tiles.get(), P.n_rank_tiles, P.world, P.world > 1 ? P.rank : -1, w, h, image, st));
            frame.launches += 1;
            return B200RT_OK;
        };
        rc = timed_launch(s, st, true, stats ? &frame : nullptr, integrate_untile, [&] { return output_stage(s, w, h, fb_out, rgba8_out, flip_y, st); });
        if (rc) return rc;
    }
    else
    {
        // N devices, one host thread each: interleaved tiles, scene replicated, mean radiance gathered on rank 0's device, where
        // `framebuffer += final; tone map` (render_kernel.cpp:169-180) happens against the incoming framebuffer
        const size_t tiles_padded = (size_t)b200rt_tiles_for_rank(w, h, 0, n_dev);
        CU(s->d_gather.grow(tiles_padded * kTilePixels * (size_t)n_dev));
        if (!fb_zero) { if ((rc = copy_to_device(s, image, fb_in, image_px * sizeof(float4), st))) return rc; h2d += image_px * sizeof(float4); }
        else CU(launch_fill_f4(image, image_px, make_float4(0.0f, 0.0f, 0.0f, 1.0f), st));
        CU(cudaStreamSynchronize(st));
        std::vector<LaunchResult> res((size_t)n_dev);
        rc = run_ranks(n_dev, [&](int d) {
            RenderParams Pd = P;
            Pd.rank = d; Pd.world = n_dev;
            Pd.n_rank_tiles = b200rt_tiles_for_rank(w, h, d, n_dev);
            Pd.flags |= B200RT_FLAG_LINEAR_TILES;
            return render_rank(d == 0 ? s : s->replicas[(size_t)d - 1], s, Pd, integrator, tiles_padded, &res[(size_t)d]);
        });
        if (rc) return rc;
        for (const LaunchResult& r : res) { frame.rays += r.rays; frame.launches += r.launches; frame.ms = std::max(frame.ms, r.ms); }
        CU(launch_untile_accumulate(s->d_gather.get(), (int)tiles_padded, n_dev, w, h, image, st));
        frame.launches += 1;
        if ((rc = output_stage(s, w, h, fb_out, rgba8_out, flip_y, st))) return rc;
    }
    if (stats)
    {
        launch_stats(frame, stats);
        stats->samples = (n_dev == 1 ? pixels_of_rank(P, w, h) : (unsigned long long)image_px) * (unsigned long long)spp;
        if ((rc = fill_kernel_times(s, stats))) return rc;
        stats->gpu_launches += rgba8_out ? 1 : 0;
        stats->h2d_bytes = h2d; stats->d2h_bytes = image_px * (rgba8_out ? 4 : sizeof(float4));
        stats->total_ms = std::chrono::duration<double, std::milli>(std::chrono::high_resolution_clock::now() - t0).count();
    }
    return B200RT_OK;
}

} // namespace

extern "C" {

int b200rt_render(b200rt_scene* s, const float* camera17, int w, int h, int spp, int bounces, float* fb,
                  const b200rt_render_options* opts, b200rt_stats* stats)
{
    if (!fb) return fail(B200RT_ERR_ARG, "framebuffer must not be NULL");
    return render_frame(s, camera17, w, h, spp, bounces, fb, fb, nullptr, 0, opts, stats);
}

int b200rt_render_rgba8(b200rt_scene* s, const float* camera17, int w, int h, int spp, int bounces, const float* fb_in_or_null,
                        int flip_y, unsigned char* out_rgba8, const b200rt_render_options* opts, b200rt_stats* stats)
{
    if (!out_rgba8) return fail(B200RT_ERR_ARG, "out_rgba8 must not be NULL");
    if (opts && opts->world > 1) return fail(B200RT_ERR_ARG, "b200rt_render_rgba8 renders whole frames (rank/world must stay 0/1)");
    return render_frame(s, camera17, w, h, spp, bounces, fb_in_or_null, nullptr, out_rgba8, flip_y, opts, stats);
}

int b200rt_render_region(b200rt_scene* s, const float* camera17, int w, int h, int spp, int bounces, int x0, int y0, int x1, int y1,
                         float* out_rgba, const b200rt_render_options* opts, b200rt_stats* stats)
{
    RenderParams P;
    int rc = make_params(s, camera17, w, h, spp, bounces, opts, P);
    if (rc) return rc;
    if (!out_rgba) return fail(B200RT_ERR_ARG, "out_rgba must not be NULL");
    if (x0 < 0 || y0 < 0 || x1 > w || y1 > h || x0 >= x1 || y0 >= y1) return fail(B200RT_ERR_ARG, "bad region [%d,%d) x [%d,%d) of %dx%d", x0, x1, y0, y1, w, h);
    if ((long long)(x1 - x0) * (y1 - y0) > (1ll << 30)) return fail(B200RT_ERR_ARG, "region too large");
    ON_DEVICE(s->device);
    const size_t px = (size_t)(x1 - x0) * (y1 - y0);
    if ((rc = ensure_scratch(s, px, 0, 0))) return rc;
    P.rank = 0; P.world = 1;
    P.flags &= ~B200RT_FLAG_LINEAR_TILES;
    P.rx0 = x0; P.ry0 = y0; P.rw = x1 - x0; P.rh = y1 - y0;
    cudaStream_t st = 0;
    SceneDev dev;
    if ((rc = launch_scene(s, P.flags, &dev))) return rc;
    LaunchResult r;
    r.launches = 1;
    // one lane per pixel through the megakernel's state machine (both integrators produce identical pixels)
    rc = timed_launch(s, st, true, stats ? &r : nullptr,
                      [&] { CU(launch_megakernel(dev, P, nullptr, s->d_tiles.get(), s->d_work.get(), s->d_rays.get(), st)); return B200RT_OK; },
                      [&] { return copy_to_host(s, out_rgba, s->d_tiles.get(), px * sizeof(float4), st); });
    if (rc || !stats) return rc;
    launch_stats(r, stats);
    stats->samples = (unsigned long long)px * (unsigned long long)spp;
    stats->h2d_bytes = 17 * sizeof(float); stats->d2h_bytes = px * sizeof(float4);
    return B200RT_OK;
}

} // extern "C"

extern "C" {

int b200rt_scene_update_triangles(b200rt_scene* s, const float* tri_xyz9, int n_tri, b200rt_stats* stats)
{
    return update_triangles(s, tri_xyz9, false, n_tri, 0, stats);
}

int b200rt_scene_update_triangles_device(b200rt_scene* s, const void* dev_tri_xyz9, int n_tri, void* cuda_stream, b200rt_stats* stats)
{
    return update_triangles(s, dev_tri_xyz9, true, n_tri, (cudaStream_t)cuda_stream, stats);
}

int b200rt_scene_get_bvh_arrays(b200rt_scene* s, int replica, void* wide80_out, float* axis16_out, float* diag16_out, float* tris12_out)
{
    if (!s) return fail(B200RT_ERR_ARG, "NULL scene");
    if (replica < 0 || replica > (int)s->replicas.size()) return fail(B200RT_ERR_ARG, "replica %d of %d", replica, 1 + (int)s->replicas.size());
    const b200rt_scene* r = replica == 0 ? s : s->replicas[(size_t)replica - 1];
    ON_DEVICE(r->device);
    const size_t n_wide = (size_t)r->info.n_wide_nodes, n_axis = (size_t)r->info.n_inner_nodes, n_tri = (size_t)r->dev.n_tri;
    if (wide80_out && n_wide) CU(cudaMemcpy(wide80_out, r->dev.wide, n_wide * sizeof(WideNode), cudaMemcpyDeviceToHost));
    if (axis16_out && n_axis) CU(cudaMemcpy(axis16_out, r->dev.axis, n_axis * sizeof(AxisNode), cudaMemcpyDeviceToHost));
    if (diag16_out && n_axis && r->dev.has_diag) CU(cudaMemcpy(diag16_out, r->dev.diag, n_axis * sizeof(DiagNode), cudaMemcpyDeviceToHost));
    if (tris12_out && n_tri) CU(cudaMemcpy(tris12_out, r->dev.tris, n_tri * sizeof(LeafTriangle), cudaMemcpyDeviceToHost));
    return B200RT_OK;
}

} // extern "C"

// An accumulator keeps, for every rank d of its scene (rank 0 = the scene, rank d = replicas[d - 1]), the generator state, the linear
// radiance sum and the mean-radiance tiles of the 16x16 tiles d owns (tile_id % n_ranks == d), tile-major, on that rank's device. A
// single-device scene has one rank that owns the whole frame. A rank owns no tile when the frame has fewer tiles than there are ranks.
struct b200rt_accum
{
    struct Rank
    {
        b200rt_scene* scene = nullptr;
        int n_tiles = 0;
        DevArray<uint32_t> d_rng; DevArray<float4> d_sum, d_tiles;
    };
    b200rt_scene* scene = nullptr;
    float camera17[17] = {};
    int w = 0, h = 0, spp_total = 0, bounces = 0, done = 0;
    std::vector<Rank> ranks;
};

namespace {

// tone_map(fb_in + mean radiance so far) into fb_out, or its RGBA8 quantisation into rgba8_out (exactly one is non-NULL). On a
// multi-device scene the ranks' tiles are first gathered into rank 0's gather buffer.
int accum_resolve(b200rt_accum* a, const float* fb_in, float* fb_out, unsigned char* rgba8_out, int flip_y)
{
    if (!a || (!fb_out && !rgba8_out)) return fail(B200RT_ERR_ARG, "NULL argument");
    if (a->done <= 0) return fail(B200RT_ERR_ARG, "nothing accumulated yet");
    b200rt_scene* s = a->scene;
    const int n_dev = (int)a->ranks.size();
    ON_DEVICE(s->device);
    const size_t image_px = (size_t)a->w * a->h;
    int rc = ensure_scratch(s, 0, image_px, 0);
    if (rc) return rc;
    const float4* gathered = a->ranks[0].d_tiles.get();
    int tiles_padded = a->ranks[0].n_tiles;
    if (n_dev > 1)
    {
        tiles_padded = b200rt_tiles_for_rank(a->w, a->h, 0, n_dev);
        CU(s->d_gather.grow((size_t)tiles_padded * kTilePixels * n_dev));
        for (int d = 0; d < n_dev; d++)
        {
            const b200rt_accum::Rank& k = a->ranks[(size_t)d];
            if ((rc = gather_rank(k.scene, s, k.d_tiles.get(), d, k.n_tiles, (size_t)tiles_padded))) return rc;
        }
        gathered = s->d_gather.get();
    }
    cudaStream_t st = 0;
    if (fb_in) { if ((rc = copy_to_device(s, s->d_image.get(), fb_in, image_px * sizeof(float4), st))) return rc; }
    else CU(launch_fill_f4(s->d_image.get(), image_px, make_float4(0.0f, 0.0f, 0.0f, 1.0f), st));
    CU(launch_untile_accumulate(gathered, tiles_padded, n_dev, a->w, a->h, s->d_image.get(), st));
    return output_stage(s, a->w, a->h, fb_out, rgba8_out, flip_y, st);
}

} // namespace

extern "C" {

int b200rt_accum_create(b200rt_scene* s, const float* camera17, int w, int h, int spp_total, int bounces, b200rt_accum** out)
{
    if (!out) return fail(B200RT_ERR_ARG, "out must not be NULL");
    *out = nullptr;
    if (!s || !camera17) return fail(B200RT_ERR_ARG, "scene and camera must not be NULL");
    if (w <= 0 || h <= 0 || spp_total <= 0 || bounces <= 0) return fail(B200RT_ERR_ARG, "bad accumulator arguments");
    ON_DEVICE(s->device);
    b200rt_accum* a = new (std::nothrow) b200rt_accum;
    if (!a) return fail(B200RT_ERR_ALLOC, "out of host memory");
    a->scene = s; a->w = w; a->h = h; a->spp_total = spp_total; a->bounces = bounces;
    std::memcpy(a->camera17, camera17, sizeof(a->camera17));
    const int n_dev = 1 + (int)s->replicas.size();
    a->ranks.resize((size_t)n_dev);
    cudaError_t e = cudaSuccess;
    for (int d = 0; d < n_dev && e == cudaSuccess; d++)
    {
        b200rt_accum::Rank& k = a->ranks[(size_t)d];
        k.scene = d == 0 ? s : s->replicas[(size_t)d - 1];
        k.n_tiles = b200rt_tiles_for_rank(w, h, d, n_dev);
        if (!k.n_tiles) continue;
        const size_t n_slots = (size_t)k.n_tiles * kTilePixels;
        DeviceScope scope(k.scene->device);
        e = scope.err;
        if (e == cudaSuccess) e = k.d_rng.grow(n_slots);
        if (e == cudaSuccess) e = k.d_sum.grow(n_slots);
        if (e == cudaSuccess) e = k.d_tiles.grow(n_slots);
        if (e == cudaSuccess) e = cudaMemset(k.d_tiles.get(), 0, n_slots * sizeof(float4));
    }
    if (e != cudaSuccess) { b200rt_accum_destroy(a); return fail(B200RT_ERR_CUDA, "accumulator allocation: %s", cudaGetErrorString(e)); }
    *out = a;
    return B200RT_OK;
}

int b200rt_accum_samples(const b200rt_accum* a) { return a ? a->done : 0; }

int b200rt_accum_add(b200rt_accum* a, int n_samples, const b200rt_render_options* opts, b200rt_stats* stats)
{
    if (!a) return fail(B200RT_ERR_ARG, "NULL accumulator");
    if (n_samples <= 0 || a->done + n_samples > a->spp_total) return fail(B200RT_ERR_ARG, "%d more samples after %d of %d", n_samples, a->done, a->spp_total);
    b200rt_scene* s = a->scene;
    RenderParams P;
    int rc = make_params(s, a->camera17, a->w, a->h, a->spp_total, a->bounces, opts, P);
    if (rc) return rc;
    if (P.world != 1) return fail(B200RT_ERR_ARG, "accumulators render whole frames (rank/world must stay 0/1)");
    const int integrator = opts ? opts->integrator : B200RT_INTEGRATOR_WAVEFRONT;
    if (integrator != B200RT_INTEGRATOR_WAVEFRONT && integrator != B200RT_INTEGRATOR_PERSISTENT)
        return fail(B200RT_ERR_ARG, "accumulators run on the wavefront or the persistent integrator");
    const int n_dev = (int)a->ranks.size();
    // checked here for every rank, so that a refused add has launched on none of them
    for (const b200rt_accum::Rank& k : a->ranks)
    {
        SceneDev unused;
        if ((rc = launch_scene(k.scene, P.flags, &unused))) return rc;
    }
    auto t0 = std::chrono::high_resolution_clock::now();
    ON_DEVICE(s->device);
    P.flags |= B200RT_FLAG_LINEAR_TILES;
    P.sample_begin = a->done; P.sample_end = a->done + n_samples;
    std::vector<LaunchResult> res((size_t)n_dev);
    // rank d continues the pixels of its own tiles from its own state; nothing crosses devices until a resolve
    auto add_rank = [&](int d) -> int {
        const b200rt_accum::Rank& k = a->ranks[(size_t)d];
        if (!k.n_tiles) return B200RT_OK;
        RenderParams Pd = P;
        Pd.rank = d; Pd.world = n_dev; Pd.n_rank_tiles = k.n_tiles;
        Pd.acc_rng = k.d_rng.get(); Pd.acc_sum = k.d_sum.get();
        cudaStream_t st = 0;                 // a single-device accumulator runs on the caller's thread and the legacy stream
        if (n_dev > 1)
        {
            const int rc_s = ensure_rank_stream(k.scene);
            if (rc_s) return rc_s;
            st = k.scene->mg_stream;
        }
        return integrate_rank(k.scene, Pd, integrator, k.d_tiles.get(), st, &res[(size_t)d]);
    };
    rc = n_dev == 1 ? add_rank(0) : run_ranks(n_dev, add_rank);
    if (rc) return rc;
    a->done += n_samples;
    if (stats)
    {
        std::memset(stats, 0, sizeof(*stats));
        float ms = 0.0f;
        for (const LaunchResult& r : res) { stats->rays += r.rays; stats->gpu_launches += r.launches; ms = std::max(ms, r.ms); }
        stats->samples = (unsigned long long)a->w * a->h * (unsigned long long)n_samples;
        stats->kernel_ms = ms;
        stats->total_ms = n_dev == 1 ? ms : std::chrono::duration<double, std::milli>(std::chrono::high_resolution_clock::now() - t0).count();
        if ((rc = fill_kernel_times(s, stats))) return rc;
    }
    return B200RT_OK;
}

int b200rt_accum_resolve(b200rt_accum* a, const float* fb_in, float* fb_out)
{
    return accum_resolve(a, fb_in, fb_out, nullptr, 0);
}

int b200rt_accum_resolve_rgba8(b200rt_accum* a, const float* fb_in, int flip_y, unsigned char* out_rgba8)
{
    if (!out_rgba8) return fail(B200RT_ERR_ARG, "out_rgba8 must not be NULL");
    return accum_resolve(a, fb_in, nullptr, out_rgba8, flip_y);
}

void b200rt_accum_destroy(b200rt_accum* a)
{
    if (!a) return;
    for (b200rt_accum::Rank& k : a->ranks)
        if (k.scene) { DeviceScope scope(k.scene->device); k = b200rt_accum::Rank{}; }      // frees the rank's arrays on its device
    delete a;
}

int b200rt_rng_stream(int x, int y, int spp, int n, uint32_t* state_out, float* floats_out)
{
    if (n < 0 || !state_out || (n > 0 && !floats_out)) return fail(B200RT_ERR_ARG, "bad rng_stream arguments");
    const int rc = require_device("b200rt");
    if (rc) return rc;
    DevArray<uint32_t> d_state; DevArray<float> d_f;
    cudaError_t e = d_state.grow(1);
    if (e == cudaSuccess) e = d_f.grow((size_t)std::max(n, 1));
    if (e == cudaSuccess) e = launch_rng_stream(x, y, spp, n, d_state.get(), d_f.get(), 0);
    if (e == cudaSuccess) e = cudaMemcpy(state_out, d_state.get(), sizeof(uint32_t), cudaMemcpyDeviceToHost);
    if (e == cudaSuccess && n) e = cudaMemcpy(floats_out, d_f.get(), sizeof(float) * (size_t)n, cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) return fail(B200RT_ERR_CUDA, "rng_stream: %s", cudaGetErrorString(e));
    return B200RT_OK;
}

int b200rt_obj_load(const char* path, b200rt_obj** out)
{
    if (!path || !out) return fail(B200RT_ERR_ARG, "NULL argument");
    *out = nullptr;
    b200rt_obj* o = new (std::nothrow) b200rt_obj;
    if (!o) return fail(B200RT_ERR_ALLOC, "out of host memory");
    std::string err;
    bool ok = false;
    try { ok = load_obj(path, o->a, err); }
    catch (const std::exception& e) { err = e.what(); }
    if (!ok) { delete o; return fail(B200RT_ERR_ARG, "OBJ ingest: %s", err.c_str()); }
    *out = o;
    return B200RT_OK;
}

int b200rt_obj_get(const b200rt_obj* o, const float** tri_xyz9, int* n_tri, const int** tri_material, const float** materials10,
                   int* n_materials, const int** emissive_tri, int* n_emissive)
{
    if (!o) return fail(B200RT_ERR_ARG, "NULL obj");
    if (tri_xyz9) *tri_xyz9 = o->a.tri_xyz9.data();
    if (n_tri) *n_tri = (int)(o->a.tri_xyz9.size() / 9);
    if (tri_material) *tri_material = o->a.tri_material.data();
    if (materials10) *materials10 = o->a.materials10.data();
    if (n_materials) *n_materials = (int)(o->a.materials10.size() / 10);
    if (emissive_tri) *emissive_tri = o->a.emissive_tri.data();
    if (n_emissive) *n_emissive = (int)o->a.emissive_tri.size();
    return B200RT_OK;
}

void b200rt_obj_destroy(b200rt_obj* o) { delete o; }

int b200rt_hdr_load(const char* path, int flip_y, b200rt_hdr** out)
{
    if (!path || !out) return fail(B200RT_ERR_ARG, "NULL argument");
    *out = nullptr;
    b200rt_hdr* h = new (std::nothrow) b200rt_hdr;
    if (!h) return fail(B200RT_ERR_ALLOC, "out of host memory");
    std::string err;
    bool ok = false;
    try { ok = load_hdr(path, flip_y != 0, h->rgb, h->w, h->h, err); }
    catch (const std::exception& e) { err = e.what(); }
    if (!ok) { delete h; return fail(B200RT_ERR_ARG, "HDR ingest: %s", err.c_str()); }
    *out = h;
    return B200RT_OK;
}

int b200rt_hdr_get(const b200rt_hdr* h, const float** rgb, int* width, int* height)
{
    if (!h) return fail(B200RT_ERR_ARG, "NULL hdr");
    if (rgb) *rgb = h->rgb.data();
    if (width) *width = h->w;
    if (height) *height = h->h;
    return B200RT_OK;
}

void b200rt_hdr_destroy(b200rt_hdr* h) { delete h; }

int b200rt_env_cdf_search(b200rt_scene* s, const float* values, int n, int use_guide, int* xy_out)
{
    if (!s || n < 0 || (n > 0 && (!values || !xy_out))) return fail(B200RT_ERR_ARG, "bad env_cdf_search arguments");
    if (n == 0) return B200RT_OK;
    ON_DEVICE(s->device);
    SceneDev dev = s->dev;
    if (!use_guide) dev.cdf_guide = nullptr;
    else if (!dev.cdf_guide) return fail(B200RT_ERR_ARG, "this scene has no CDF guide table (the running sum is not monotone, or B200RT_CDF_GUIDE=0)");
    DevArray<float> d_v; DevArray<int> d_xy;
    cudaError_t e = d_v.grow((size_t)n);
    if (e == cudaSuccess) e = d_xy.grow(2 * (size_t)n);
    if (e == cudaSuccess) e = cudaMemcpy(d_v.get(), values, sizeof(float) * (size_t)n, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = launch_env_cdf_search(dev, d_v.get(), n, d_xy.get(), 0);
    if (e == cudaSuccess) e = cudaMemcpy(xy_out, d_xy.get(), sizeof(int) * 2 * (size_t)n, cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) return fail(B200RT_ERR_CUDA, "env_cdf_search: %s", cudaGetErrorString(e));
    return B200RT_OK;
}

int b200rt_host_alloc(size_t bytes, void** out)
{
    if (!out) return fail(B200RT_ERR_ARG, "out must not be NULL");
    *out = nullptr;
    CU(cudaMallocHost(out, std::max<size_t>(bytes, 1)));
    return B200RT_OK;
}

void b200rt_host_free(void* p) { if (p) cudaFreeHost(p); }

int b200rt_untile_accumulate_device(b200rt_scene* s, const void* dev_gathered, int tiles_per_rank_padded, int world, int w, int h,
                                    void* dev_fb_inout, void* cuda_stream)
{
    if (!s || !dev_gathered || !dev_fb_inout || world <= 0 || w <= 0 || h <= 0) return fail(B200RT_ERR_ARG, "bad untile arguments");
    if (tiles_per_rank_padded < b200rt_tiles_for_rank(w, h, 0, world)) return fail(B200RT_ERR_ARG, "tiles_per_rank_padded too small");
    ON_DEVICE(s->device);
    CU(launch_untile_accumulate((const float4*)dev_gathered, tiles_per_rank_padded, world, w, h, (float4*)dev_fb_inout, (cudaStream_t)cuda_stream));
    return B200RT_OK;
}

int b200rt_quantise_rgba8_device(const void* dev_image_rgba, int w, int h, int flip_y, void* dev_out_rgba8, void* cuda_stream)
{
    if (!dev_image_rgba || !dev_out_rgba8 || w <= 0 || h <= 0) return fail(B200RT_ERR_ARG, "bad quantise arguments");
    CU(launch_quantise_rgba8((const float4*)dev_image_rgba, w, h, flip_y, dev_out_rgba8, (cudaStream_t)cuda_stream));
    return B200RT_OK;
}

int b200rt_quantise_rgba8(const float* image_rgba, int w, int h, int flip_y, unsigned char* out_rgba8)
{
    if (!image_rgba || !out_rgba8 || w <= 0 || h <= 0) return fail(B200RT_ERR_ARG, "bad quantise arguments");
    const int rc = require_device("b200rt");
    if (rc) return rc;
    const size_t px = (size_t)w * h;
    DevArray<float4> d_in; DevArray<unsigned char> d_out;
    cudaError_t e = d_in.grow(px);
    if (e == cudaSuccess) e = d_out.grow(px * 4);
    if (e == cudaSuccess) e = cudaMemcpy(d_in.get(), image_rgba, px * sizeof(float4), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = launch_quantise_rgba8(d_in.get(), w, h, flip_y, d_out.get(), 0);
    if (e == cudaSuccess) e = cudaMemcpy(out_rgba8, d_out.get(), px * 4, cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) return fail(B200RT_ERR_CUDA, "quantise_rgba8: %s", cudaGetErrorString(e));
    return B200RT_OK;
}

int b200rt_denoise_guided(const float* image, int channels, const float* albedo, const float* normal, int w, int h, float blend,
                          int iterations, float sigma, float* out)
{
    if (!image || !out || w <= 0 || h <= 0 || (channels != 3 && channels != 4)) return fail(B200RT_ERR_ARG, "bad denoise arguments");
    const int rc = require_device("b200rt");
    if (rc) return rc;
    if (iterations <= 0) iterations = 5;
    if (iterations > 8) iterations = 8;
    if (!(sigma > 0.0f)) sigma = 0.45f;
    const size_t n = (size_t)w * h * channels, n_guide = (size_t)w * h * 3;
    DevArray<float> d_in, d_tmp, d_out, d_albedo, d_normal;
    cudaError_t e = d_in.grow(n);
    if (e == cudaSuccess) e = d_tmp.grow(n);
    if (e == cudaSuccess) e = d_out.grow(n);
    if (e == cudaSuccess && albedo) e = d_albedo.grow(n_guide);
    if (e == cudaSuccess && normal) e = d_normal.grow(n_guide);
    if (e == cudaSuccess) e = cudaMemcpy(d_in.get(), image, n * sizeof(float), cudaMemcpyHostToDevice);
    if (e == cudaSuccess && albedo) e = cudaMemcpy(d_albedo.get(), albedo, n_guide * sizeof(float), cudaMemcpyHostToDevice);
    if (e == cudaSuccess && normal) e = cudaMemcpy(d_normal.get(), normal, n_guide * sizeof(float), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = launch_denoise(d_in.get(), channels, d_albedo.get(), d_normal.get(), w, h, iterations, sigma, blend, d_tmp.get(), d_out.get(), 0);
    if (e == cudaSuccess) e = cudaMemcpy(out, d_out.get(), n * sizeof(float), cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) return fail(B200RT_ERR_CUDA, "denoise: %s", cudaGetErrorString(e));
    return B200RT_OK;
}

int b200rt_denoise(const float* image, int channels, int w, int h, float blend, int iterations, float sigma, float* out)
{
    return b200rt_denoise_guided(image, channels, nullptr, nullptr, w, h, blend, iterations, sigma, out);
}

int b200rt_render_aovs_device(b200rt_scene* s, const float* camera17, int w, int h, int samples_per_axis, void* dev_albedo, void* dev_normal,
                              const b200rt_render_options* opts, void* cuda_stream, b200rt_stats* stats)
{
    RenderParams P;
    int rc = make_params(s, camera17, w, h, 1, 1, opts, P);
    if (rc) return rc;
    if (samples_per_axis < 1 || samples_per_axis > 16) return fail(B200RT_ERR_ARG, "samples_per_axis %d outside 1..16", samples_per_axis);
    if (!dev_albedo && !dev_normal) return fail(B200RT_ERR_ARG, "at least one of the albedo / normal outputs must be given");
    if (P.world != 1) return fail(B200RT_ERR_ARG, "feature buffers are computed for whole frames (rank/world must stay 0/1)");
    ON_DEVICE(s->device);
    if ((rc = ensure_scratch(s, 0, 0, 0))) return rc;
    cudaStream_t st = (cudaStream_t)cuda_stream;
    LaunchResult r;
    r.launches = 1;
    rc = timed_launch(s, st, false, stats ? &r : nullptr,
                      [&] { CU(launch_aov(s->dev, P, samples_per_axis, (float*)dev_albedo, (float*)dev_normal, st)); return B200RT_OK; });
    if (rc || !stats) return rc;
    launch_stats(r, stats);
    stats->rays = stats->samples = (unsigned long long)w * h * samples_per_axis * samples_per_axis;
    return B200RT_OK;
}

int b200rt_render_aovs(b200rt_scene* s, const float* camera17, int w, int h, int samples_per_axis, float* albedo_out, float* normal_out,
                       const b200rt_render_options* opts, b200rt_stats* stats)
{
    if (!s) return fail(B200RT_ERR_ARG, "NULL scene");
    if (!albedo_out && !normal_out) return fail(B200RT_ERR_ARG, "at least one of the albedo / normal outputs must be given");
    if (w <= 0 || h <= 0) return fail(B200RT_ERR_ARG, "bad frame size");
    auto t0 = std::chrono::high_resolution_clock::now();
    ON_DEVICE(s->device);
    const size_t n = (size_t)w * h * 3, bytes = n * sizeof(float);
    DevArray<float> d_albedo, d_normal;
    cudaError_t e = cudaSuccess;
    if (albedo_out) e = d_albedo.grow(n);
    if (e == cudaSuccess && normal_out) e = d_normal.grow(n);
    if (e != cudaSuccess) return fail(B200RT_ERR_CUDA, "render_aovs: %s", cudaGetErrorString(e));
    int rc = b200rt_render_aovs_device(s, camera17, w, h, samples_per_axis, d_albedo.get(), d_normal.get(), opts, nullptr, stats);
    if (rc) return rc;
    if (albedo_out && (rc = copy_to_host(s, albedo_out, d_albedo.get(), bytes, 0))) return rc;
    if (normal_out && (rc = copy_to_host(s, normal_out, d_normal.get(), bytes, 0))) return rc;
    if (stats)
    {
        stats->d2h_bytes = (albedo_out ? bytes : 0) + (normal_out ? bytes : 0); stats->h2d_bytes = 17 * sizeof(float);
        stats->total_ms = std::chrono::duration<double, std::milli>(std::chrono::high_resolution_clock::now() - t0).count();
    }
    return B200RT_OK;
}

int b200rt_trace_primary_device(b200rt_scene* s, const float* camera17, int w, int h, int sample, int spp_for_seed,
                                void* dev_prim, void* dev_t, const b200rt_render_options* opts, void* cuda_stream, b200rt_stats* stats)
{
    RenderParams P;
    int rc = make_params(s, camera17, w, h, spp_for_seed, 1, opts, P);
    if (rc) return rc;
    if (!dev_prim || !dev_t) return fail(B200RT_ERR_ARG, "output buffers must not be NULL");
    if (sample > 0) return fail(B200RT_ERR_ARG, "only sample 0 (or < 0 = un-jittered) has a path-independent camera ray");
    ON_DEVICE(s->device);
    if ((rc = ensure_scratch(s, 0, 0, 0))) return rc;
    cudaStream_t st = (cudaStream_t)cuda_stream;
    LaunchResult r;
    r.launches = 1;
    rc = timed_launch(s, st, false, stats ? &r : nullptr,
                      [&] { CU(launch_primary(s->dev, P, sample, (int*)dev_prim, (float*)dev_t, st)); return B200RT_OK; });
    if (rc || !stats) return rc;
    launch_stats(r, stats);
    stats->rays = stats->samples = pixels_of_rank(P, w, h);
    return B200RT_OK;
}

int b200rt_trace_primary(b200rt_scene* s, const float* camera17, int w, int h, int sample, int spp_for_seed,
                         int* prim_out, float* t_out, const b200rt_render_options* opts, b200rt_stats* stats)
{
    if (!s) return fail(B200RT_ERR_ARG, "NULL scene");
    if (!prim_out || !t_out) return fail(B200RT_ERR_ARG, "output buffers must not be NULL");
    if (w <= 0 || h <= 0) return fail(B200RT_ERR_ARG, "bad frame size");
    auto t0 = std::chrono::high_resolution_clock::now();
    ON_DEVICE(s->device);
    const size_t px = (size_t)w * h;
    int rc = ensure_scratch(s, 0, 0, px);
    if (rc) return rc;
    if (opts && opts->world > 1)
    {
        // pixels of other ranks read as "miss"; a whole-frame call writes every pixel itself
        CU(cudaMemsetAsync(s->d_prim.get(), 0xff, px * sizeof(int), 0));
        CU(launch_fill_f32(s->d_t.get(), px, -1.0f, 0));
    }
    rc = b200rt_trace_primary_device(s, camera17, w, h, sample, spp_for_seed, s->d_prim.get(), s->d_t.get(), opts, nullptr, stats);
    if (rc) return rc;
    if ((rc = copy_to_host(s, prim_out, s->d_prim.get(), px * sizeof(int), 0))) return rc;
    if ((rc = copy_to_host(s, t_out, s->d_t.get(), px * sizeof(float), 0))) return rc;
    if (stats)
    {
        stats->d2h_bytes = px * 8; stats->h2d_bytes = 17 * sizeof(float);
        stats->total_ms = std::chrono::duration<double, std::milli>(std::chrono::high_resolution_clock::now() - t0).count();
    }
    return B200RT_OK;
}

int b200rt_trace_rays_device(b200rt_scene* s, const void* dev_rays6, int n, int any_hit, void* dev_prim, void* dev_t, void* dev_extra8,
                             const b200rt_render_options* opts, void* cuda_stream, b200rt_stats* stats)
{
    if (!s) return fail(B200RT_ERR_ARG, "NULL scene");
    if (n < 0 || (n > 0 && (!dev_rays6 || !dev_prim || !dev_t))) return fail(B200RT_ERR_ARG, "bad ray buffers");
    ON_DEVICE(s->device);
    int rc = ensure_scratch(s, 0, 0, 0);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)cuda_stream;
    LaunchResult r;
    r.launches = 1;
    rc = timed_launch(s, st, false, stats ? &r : nullptr, [&] {
        CU(launch_trace_rays(s->dev, (const float*)dev_rays6, n, any_hit, opts ? opts->flags : 0, (int*)dev_prim, (float*)dev_t, (float*)dev_extra8, st));
        return B200RT_OK;
    });
    if (rc || !stats) return rc;
    launch_stats(r, stats);
    stats->rays = (unsigned long long)n;
    return B200RT_OK;
}

int b200rt_trace_rays(b200rt_scene* s, const float* rays6, int n, int any_hit, int* prim_out, float* t_out, float* extra8,
                      const b200rt_render_options* opts)
{
    if (!s) return fail(B200RT_ERR_ARG, "NULL scene");
    if (n < 0 || (n > 0 && (!rays6 || !prim_out || !t_out))) return fail(B200RT_ERR_ARG, "bad ray buffers");
    if (n == 0) return B200RT_OK;
    ON_DEVICE(s->device);
    DevArray<float> d_rays6, d_t, d_extra; DevArray<int> d_prim;
    cudaError_t e = d_rays6.grow(6 * (size_t)n);
    if (e == cudaSuccess) e = d_prim.grow((size_t)n);
    if (e == cudaSuccess) e = d_t.grow((size_t)n);
    if (e == cudaSuccess && extra8) e = d_extra.grow(8 * (size_t)n);
    if (e == cudaSuccess) e = cudaMemcpy(d_rays6.get(), rays6, sizeof(float) * 6 * (size_t)n, cudaMemcpyHostToDevice);
    if (e != cudaSuccess) return fail(B200RT_ERR_CUDA, "trace_rays: %s", cudaGetErrorString(e));
    const int rc = b200rt_trace_rays_device(s, d_rays6.get(), n, any_hit, d_prim.get(), d_t.get(), d_extra.get(), opts, nullptr, nullptr);
    if (rc) return rc;
    e = cudaMemcpy(prim_out, d_prim.get(), sizeof(int) * (size_t)n, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess) e = cudaMemcpy(t_out, d_t.get(), sizeof(float) * (size_t)n, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess && extra8) e = cudaMemcpy(extra8, d_extra.get(), sizeof(float) * 8 * (size_t)n, cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) return fail(B200RT_ERR_CUDA, "trace_rays: %s", cudaGetErrorString(e));
    return B200RT_OK;
}

} // extern "C"
