// K3: wavefront integrator with path regeneration (sm_100a). Compiled with -fmad=false (see pt_device.cuh).
//
// One slot per pixel of this rank's tile-major buffer. A slot carries the pixel's xorshift state through all of its
// samples, so the per-pixel RNG stream is consumed in exactly the reference's order (render_kernel.cpp:75-181) and the
// image is bit-identical to the megakernel's. Every iteration is two launches:
//
//   wf_shade : per slot — resolve the side rays of the previous surface interaction (sample_color += (light + env) *
//              throughput, :128), consume the path ray's closest hit (miss -> sky/finish sample, hit -> material fetch,
//              the four side rays of sample_light_sources / sample_environment_map with their MIS weights, the
//              continuation sample, termination tests :130-135), finish samples / pixels, regenerate camera rays, and
//              append every ray it produced to a compacted queue (grouped by ray kind per warp, so 32 consecutive queue
//              entries are the same kind of ray from neighbouring pixels).
//   wf_trace : persistent CTAs walk the queue; one ray per lane; closest-hit, any-hit or shadow traversal by ray kind.
//
// No RNG draw depends on a trace result (SURVEY a5), which is what allows a whole surface interaction — all four side
// rays and the continuation ray — to be generated in one shade pass and traced in one trace pass.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <utility>
#include <vector>

#include "wf_device.cuh"

namespace b200rt {

#ifndef WF_SHADE_BLOCK
#define WF_SHADE_BLOCK 256              // threads per wf_shade CTA
#endif
#ifndef WF_SHADE_MIN_BLOCKS
#define WF_SHADE_MIN_BLOCKS (1024 / WF_SHADE_BLOCK)      // 64 registers
#endif

__global__ void __launch_bounds__(256) wf_init(SceneDev S, RenderParams P, WfBuffers B, const float4* __restrict__ fb_in_rowmajor,
                                               float4* __restrict__ out_tiles)
{
    const int slot = blockIdx.x * blockDim.x + threadIdx.x;
    bool q_path = false;
    if (slot < B.n_slots)
    {
        int x, y;
        const bool inside = wf_slot_pixel(P, slot, x, y);
        if (!inside) { out_tiles[wf_out_index(B, slot)] = make_float4(0.0f, 0.0f, 0.0f, 0.0f); B.flags[slot] = WF_DONE; }
        else if (P.sample_end <= P.sample_begin || P.max_bounces <= 0)
        {
            const float n = (float)P.spp;
            out_tiles[wf_out_index(B, slot)] = pixel_output(P.flags, fb_in_rowmajor, (size_t)y * P.cam.w + x, CO(0.0f / n, 0.0f / n, 0.0f / n));
            B.flags[slot] = WF_DONE;
        }
        else
        {
            wf_begin_pixel(P, B, slot, x, y, wf_out_index(B, slot));
            q_path = true;
        }
    }
    const unsigned int active = __ballot_sync(0xffffffffu, q_path);
    if ((threadIdx.x & 31) == 0 && active) atomicAdd(&B.counters[2], (unsigned int)__popc(active));
    wf_enqueue(B.queue, &B.counters[3], q_path, ((unsigned int)slot << 3) | 4u);
}

__global__ void __launch_bounds__(WF_SHADE_BLOCK, WF_SHADE_MIN_BLOCKS) wf_shade(SceneDev S, RenderParams P, WfBuffers B, const float4* __restrict__ fb_in_rowmajor,
                                                float4* __restrict__ out_tiles, int parity)
{
    const int slot = blockIdx.x * blockDim.x + threadIdx.x;
    const int n = B.n_slots;
    unsigned int* q_count = &B.counters[3 + parity];
    if (slot == 0)
    {
        B.counters[3 + (parity ^ 1)] = 0;      // the other queue was fully consumed by the previous trace pass
        B.counters[5 + parity] = 0;            // head of the queue this pass fills
    }
    ShadeOut R;
    R.q_path = R.q0 = R.q1 = R.q2 = R.q3 = R.pixel_done = false; R.flags = 0;
    const int flags_in = slot < n ? B.flags[slot] : WF_DONE;
    if (!(flags_in & WF_DONE))
    {
        int x, y;
        wf_slot_pixel(P, slot, x, y);
        R = wf_shade_slot(S, P, B, slot, flags_in, x, y, wf_out_index(B, slot), fb_in_rowmajor, out_tiles);
    }
    const unsigned int done_mask = __ballot_sync(0xffffffffu, R.pixel_done);
    if ((threadIdx.x & 31) == 0 && done_mask) atomicSub(&B.counters[2], (unsigned int)__popc(done_mask));
    const unsigned int s3 = (unsigned int)slot << 3;
    const bool q[5] = { R.q_path, R.q0, R.q1, R.q2, R.q3 };
    const unsigned int entry[5] = { s3 | 4u, s3 | 0u, s3 | 1u, s3 | 2u, s3 | 3u };
    wf_enqueue5(B.queue, q_count, q, entry);
}

// ablation variant (B200RT_FLAG_SIMPLE_TRACE): one ray per lane, grid-stride over the queue (the warp waits for its slowest ray)
template <int TL>
__global__ void wf_trace_simple(SceneDev S, WfBuffers B, int parity)
{
    const unsigned int n_rays = B.counters[3 + parity];
    if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(B.rays_total, (unsigned long long)n_rays);
    const int n = B.n_slots;
    for (unsigned int i = blockIdx.x * blockDim.x + threadIdx.x; i < n_rays; i += gridDim.x * blockDim.x)
    {
        const unsigned int e = B.queue[i];
        const int slot = (int)(e >> 3), k = (int)(e & 7u);
        const size_t r = (size_t)k * n + slot;
        const float4 ro4 = B.ray_o[r], rd4 = B.ray_d[r];
        const int kind = __float_as_int(rd4.w);
        const int mode = kind == SIDE_SHADOW ? TRACE_SHADOW : (kind == SIDE_CLOSEST_LIGHT ? TRACE_CLOSEST : TRACE_ANY);
        Hit h;
        const bool found = trace_ray<TL>(S, V(ro4.x, ro4.y, ro4.z), V(rd4.x, rd4.y, rd4.z), ro4.w, mode, h);
        wf_store_result(B, r, mode, found, h);
    }
}

// phase-vote persistent kernel (the default on the binary layout): every lane owns one traversal state; whenever at least
// kRefillThreshold lanes of a warp are idle they are refilled with new rays from the warp's private block of the queue (blocks
// of kWarpBlock rays are claimed with one atomic), so no lane waits for the slowest ray of its warp (Aila & Laine's persistent
// threads, per lane).
#ifndef WF_LEAF_MIN
#define WF_LEAF_MIN 4
#endif
#ifdef WF_TRACE_MIN_BLOCKS
#define WF_TRACE_BOUNDS __launch_bounds__(128, WF_TRACE_MIN_BLOCKS)
#else
#define WF_TRACE_BOUNDS
#endif
constexpr int kLeafThreshold = WF_LEAF_MIN;

// one interface over the binary and the 8-ary traversal state machines, so the persistent kernel below serves every layout
template <int TL>
struct TravOps
{
    typedef Trav State;
    typedef TravStack Stack;
    static __device__ __forceinline__ void init(State& T, v3 o, v3 d, float tmax, int mode) { trav_init<TL == TL_DIAG>(T, o, d, tmax, mode); }
    static __device__ __forceinline__ bool at_node(const State& T) { return T.cur >= 0; }
    static __device__ __forceinline__ void node(const SceneDev& S, State& T, Stack& K) { trav_inner<TL == TL_DIAG>(S, T, K); }
    static __device__ __forceinline__ void leaf(const SceneDev& S, State& T, Stack& K) { trav_leaf(S, T, K); }
};
template <>
struct TravOps<TL_WIDE>
{
    typedef Trav8 State;
    typedef TravStack8 Stack;
    static __device__ __forceinline__ void init(State& T, v3 o, v3 d, float tmax, int mode) { trav8_init(T, o, d, tmax, mode); }
    static __device__ __forceinline__ bool at_node(const State& T) { return trav8_has_node(T); }
    static __device__ __forceinline__ void node(const SceneDev& S, State& T, Stack& K) { trav8_node(S, T, K); }
    static __device__ __forceinline__ void leaf(const SceneDev& S, State& T, Stack& K) { trav8_tris(S, T, K); }
};

template <int TL>
__global__ void WF_TRACE_BOUNDS wf_trace(SceneDev S, WfBuffers B, int parity)
{
    typedef TravOps<TL> Ops;
    const unsigned int FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const unsigned int n_rays = B.counters[3 + parity];
    unsigned int* head = &B.counters[5 + parity];
    if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(B.rays_total, (unsigned long long)n_rays);
    const int n = B.n_slots;
    const bool spheres = S.n_spheres != 0;
    // rays claimed per atomic: kWarpBlock when the queue is long, down to one warp's worth when it is short (otherwise a
    // few warps would serialise a short queue while the rest of the machine idles)
    const unsigned int total_warps = gridDim.x * (blockDim.x >> 5);
    const unsigned int warp_block = min((unsigned int)kWarpBlock, max(32u, (n_rays / total_warps) & ~31u));

    typename Ops::State T;
    typename Ops::Stack K;
    T.done = true;
    bool active = false;
    size_t r = 0;
    int mode = TRACE_CLOSEST;
    unsigned int blk_next = 0, blk_end = 0;       // warp-uniform: the warp's private block of queue entries
    bool exhausted = false;                       // warp-uniform: the queue has no more blocks

    for (;;)
    {
        unsigned int idle = __ballot_sync(FULL, !active);
        if (idle)
        {
            if (!exhausted && (idle == FULL || __popc(idle) >= kRefillThreshold))
            {
                if (blk_next >= blk_end)
                {
                    unsigned int b = 0;
                    if (lane == 0) b = atomicAdd(head, warp_block);
                    b = __shfl_sync(FULL, b, 0);
                    if (b >= n_rays) exhausted = true;
                    else { blk_next = b; blk_end = min(b + warp_block, n_rays); }
                }
                if (blk_next < blk_end)
                {
                    const unsigned int idx = blk_next + __popc(idle & ((1u << lane) - 1u));
                    if (!active && idx < blk_end)
                    {
                        const unsigned int e = B.queue[idx];
                        const int slot = (int)(e >> 3), k = (int)(e & 7u);
                        r = (size_t)k * n + slot;
                        const float4 ro4 = B.ray_o[r], rd4 = B.ray_d[r];
                        const int kind = __float_as_int(rd4.w);
                        mode = kind == SIDE_SHADOW ? TRACE_SHADOW : (kind == SIDE_CLOSEST_LIGHT ? TRACE_CLOSEST : TRACE_ANY);
                        Ops::init(T, V(ro4.x, ro4.y, ro4.z), V(rd4.x, rd4.y, rd4.z), ro4.w, spheres ? TRACE_CLOSEST : mode);
                        active = true;
                    }
                    blk_next = min(blk_next + (unsigned int)__popc(idle), blk_end);
                }
                idle = __ballot_sync(FULL, !active);
            }
        }
        // warp-level phase vote: all lanes that hold an inner node step together, or all lanes that hold a leaf run the
        // exact triangle tests together, whichever is the majority — the two kinds of work never interleave inside a warp
        const bool has_inner = active && Ops::at_node(T), has_leaf = active && !Ops::at_node(T);
        const unsigned int m_inner = __ballot_sync(FULL, has_inner), m_leaf = __ballot_sync(FULL, has_leaf);
        if (!(m_inner | m_leaf))
        {
            if (exhausted) break;
            continue;
        }
        if (m_inner && __popc(m_leaf) < max(__popc(m_inner), kLeafThreshold)) { if (has_inner) Ops::node(S, T, K); }
        else if (has_leaf) Ops::leaf(S, T, K);
        if (active && T.done)
        {
            bool found = T.hit.t > 0.0f;
            if (spheres) found = finish_with_spheres(S, T.o, T.d, T.tmax, mode, T.hit);
            wf_store_result(B, r, mode, found, T.hit);
            active = false;
        }
    }
}

// ---- default trace kernel for the 8-ary layout: persistent lanes + warp-cooperative triangle tests (wf_device.cuh) ------------------
#ifndef WF_COOP_MIN_BLOCKS
#define WF_COOP_MIN_BLOCKS 7            // <= 72 registers: 28 warps per SM; 32 (64 registers) measured the same, 16 (117 registers) 20 % slower
#endif
__global__ void __launch_bounds__(32 * kCoopMaxWarps, WF_COOP_MIN_BLOCKS) wf_trace_coop(SceneDev S, WfBuffers B, int parity)
{
    __shared__ CoopWarp s_warps[kCoopMaxWarps];
    CoopWarp& W = s_warps[threadIdx.x >> 5];
    const unsigned int n_rays = B.counters[3 + parity];
    if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(B.rays_total, (unsigned long long)n_rays);
    // rays claimed per atomic: kWarpBlock when the queue is long, down to one warp's worth when it is short (otherwise a
    // few warps would serialise a short queue while the rest of the machine idles)
    const unsigned int total_warps = gridDim.x * (blockDim.x >> 5);
    CoopQueueShared src;
    src.head = &B.counters[5 + parity];
    src.n_rays = n_rays;
    src.warp_block = min((unsigned int)kWarpBlock, max(32u, (n_rays / total_warps) & ~31u));
#ifdef WF_COOP_LOCAL_STACK
    TravStack8 K;
#else
    __shared__ uint2 s_stack[kSharedStackDepth * 32 * kCoopMaxWarps];
    TravStack8Shared K;
    K.sh = s_stack + threadIdx.x; K.stride = 32 * kCoopMaxWarps;
#endif
    coop_trace_queue(S, B, B.queue, src, W, K);
}

// ---- host driver ---------------------------------------------------------------------------------------------------------------
// The frame's pixels are split into n_groups interleaved tile groups (group g of rank r behaves like rank r + g * world of
// a world * n_groups partition). Each group runs its own trace/shade iteration chain on its own stream, so while one
// group's trace pass drains its longest rays (a single ray is a dependent chain of node fetches; the slowest ray of a
// pass bounds that pass) the other groups' kernels fill the machine. Groups never exchange data.
cudaError_t run_wavefront(const SceneDev& S, const RenderParams& P, const WfGroup* groups, int n_groups, const float4* fb_in_rowmajor,
                          float4* out_tiles, cudaStream_t stream, cudaEvent_t fork_event, int* launches_out, double* kernel_times4,
                          unsigned int* unfinished_out, WfTimeline* timeline)
{
    const int n_sm = current_sm_count();
    int launches = 0;
    const int tl = traversal_layout(S, P.flags);
    const bool simple = (P.flags & B200RT_FLAG_SIMPLE_TRACE) != 0;
    static const int tb_env = []() { const char* e = getenv("B200RT_TRACE_BLOCK"); int v = e ? atoi(e) : 128; return (v == 64 || v == 128 || v == 256) ? v : 128; }();
    int per_sm = 0;
    typedef void (*TraceKernel)(SceneDev, WfBuffers, int);
    static const TraceKernel kernels[2][3] = { { wf_trace<TL_AXIS>, wf_trace<TL_DIAG>, wf_trace<TL_WIDE> },
                                               { wf_trace_simple<TL_AXIS>, wf_trace_simple<TL_DIAG>, wf_trace_simple<TL_WIDE> } };
    static const bool vote_wide = []() { const char* e = getenv("B200RT_WIDE_TRACE"); return e && e[0] == 'v'; }();   // ablation: phase-vote kernel on the 8-ary layout
    const bool coop = tl == TL_WIDE && !simple && !vote_wide;
    const TraceKernel trace_kernel = coop ? wf_trace_coop : kernels[simple ? 1 : 0][tl];
    const int tb = coop ? 32 * kCoopMaxWarps : tb_env;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, trace_kernel, tb, 0);
    if (per_sm <= 0) per_sm = 1;
    // With several tile groups in flight a persistent trace kernel takes only ~4/7 of the CTAs that fit (B200RT_TRACE_GRID_PCT,
    // default 58): the rest of every SM stays free for the other groups' trace / shade kernels, which then overlap with the
    // whole pass instead of only with its tail (C3, 32 spp: 2 179 vs 2 108 Mrays/s; 72 %: 2 157, 43 %: 2 112).
    static const int grid_pct_env = []() { const char* e = getenv("B200RT_TRACE_GRID_PCT"); int v = e ? atoi(e) : 0; return v > 100 ? 100 : v; }();
    const bool timing_mode = getenv("B200RT_WF_TIMING") != nullptr || (P.flags & B200RT_FLAG_TIME_KERNELS);      // kernels run one at a time: full grid
    const int grid_pct = grid_pct_env >= 10 ? grid_pct_env : ((n_groups > 1 && !timing_mode) ? 58 : 100);
    const int trace_grid = n_sm * std::max(1, (per_sm * grid_pct + 50) / 100);
    static const bool timing_env = getenv("B200RT_WF_TIMING") != nullptr;  // diagnostics: per-kernel times on stderr (serialises the groups)
    const bool timing = timing_env || (P.flags & B200RT_FLAG_TIME_KERNELS);
    WfTimeline* const tln = (!timing && (P.flags & B200RT_FLAG_TIME_INLINE)) ? timeline : nullptr;
    if (tln)
    {
        tln->reset();
        if (!tln->origin) cudaEventCreate(&tln->origin);
        cudaEventRecord(tln->origin, stream);
    }
    int n_trace = 0, n_shade = 0;
    cudaError_t e;

    // fork: every group stream starts after the work already queued on the caller's stream. From here on an error does not
    // return: it ends the launching and falls through to the join, so that no group stream is left forked.
    if ((e = cudaEventRecord(fork_event, stream)) != cudaSuccess) return e;
    cudaError_t err = cudaSuccess;
#define WF_TRY(expr) do { if (err == cudaSuccess) { const cudaError_t e__ = (expr); if (e__ != cudaSuccess) err = e__; } } while (0)
    struct GroupRun { RenderParams P; int parity; bool finished, forked; int slot_grid; long long it, poll_it; bool poll_pending; unsigned int tail_below; };
    // barrier-free tail (persist.cu): when a group has at most B200RT_WF_TAIL_PCT % of its pixels (and at most B200RT_WF_TAIL_CAP) left,
    // or is smaller than B200RT_WF_TAIL_MIN pixels to begin with. 8-ary layout, default trace kernel only; not in the per-kernel timing modes.
    // Measured on C3 at 64 spp (profiles/r2_tail.jsonl): whole frame 433.3 ms without, 428.9 with a 30 k cap (445 with 100 k: the tail
    // kernel's throughput is below the pass kernels', it only pays once passes are latency-bound); one rank of 8: 108.1 -> 101.7 ms at 20 %.
    // (the knobs are read per frame: tools/tail_bench.py sweeps them inside one process)
    auto env_ll = [](const char* name, long long dflt) { const char* e = getenv(name); return e ? atoll(e) : dflt; };
    const int tail_pct = (int)std::min(100ll, std::max(0ll, env_ll("B200RT_WF_TAIL_PCT", 20)));
    const long long tail_cap = env_ll("B200RT_WF_TAIL_CAP", 30000);
    const int tail_min = (int)env_ll("B200RT_WF_TAIL_MIN", 16384);
    const bool passes_only = (P.flags & B200RT_FLAG_WF_PASSES_ONLY) != 0;
    const bool tail_ok = coop && tail_pct > 0 && !timing && !passes_only;
    const int tail_ctas = tail_ok ? std::max(1, wavefront_tail_max_ctas() / n_groups) : 0;
    // launches the tail that finishes group g behind whatever is queued on its stream
    auto finish_group = [&](int g, const RenderParams& GP) -> cudaError_t
    {
        const WfGroup& G = groups[g];
        WfTimeline::Launch tlt = { g, 0, 0, 0 };
        if (tln) { tlt.e0 = tln->used; cudaEventRecord(tln->take(), G.stream); }
        const cudaError_t fe = launch_wavefront_tail(S, GP, G.buf, tail_ctas, fb_in_rowmajor, out_tiles, G.stream);
        if (tln) { tlt.e1 = tln->used; cudaEventRecord(tln->take(), G.stream); tln->tails.push_back(tlt); }
        launches += 2;
        return fe;
    };
    GroupRun run[kMaxWfGroups];
    for (int g = 0; g < n_groups; g++)
    {
        const WfGroup& G = groups[g];
        GroupRun& R = run[g];
        R.P = P;
        R.P.rank = P.rank + g * P.world;
        R.P.world = P.world * n_groups;
        R.P.n_rank_tiles = G.buf.n_slots / kTilePixels;
        R.parity = 0; R.it = 0; R.poll_it = 0; R.poll_pending = false; R.forked = false;
        R.slot_grid = (G.buf.n_slots + 255) / 256;
        R.finished = R.slot_grid <= 0;
        if (err != cudaSuccess) { R.finished = true; continue; }
        WF_TRY(cudaStreamWaitEvent(G.stream, fork_event, 0));
        if (err != cudaSuccess) { R.finished = true; continue; }
        R.forked = true;
        // an empty group (fewer tiles than groups) still gets its counters cleared: the frame's ray count sums every group
        WF_TRY(cudaMemsetAsync(G.buf.counters, 0, 8 * sizeof(unsigned int), G.stream));
        WF_TRY(cudaMemsetAsync(G.buf.rays_total, 0, sizeof(unsigned long long), G.stream));
        if (R.finished) continue;
        wf_init<<<R.slot_grid, 256, 0, G.stream>>>(S, R.P, G.buf, fb_in_rowmajor, out_tiles);
        launches++;
        R.tail_below = (unsigned int)std::min<long long>(tail_cap, (long long)G.buf.n_slots * tail_pct / 100);
        if (tail_ok && G.buf.n_slots <= tail_min)
        {
            // a group this small is latency-bound from its first pass on: barrier-free from the start
            WF_TRY(finish_group(g, R.P));
            R.finished = true;
        }
    }
    const long long max_iters = (long long)(P.sample_end - P.sample_begin) * (P.max_bounces + 1) + 2;
    cudaEvent_t tev[3] = { nullptr, nullptr, nullptr };
    double t_trace = 0.0, t_shade = 0.0;
    if (timing) for (int i = 0; i < 3; i++) cudaEventCreate(&tev[i]);
    int remaining = 0;
    unsigned int unfinished = 0;
    for (int g = 0; g < n_groups; g++) remaining += run[g].finished ? 0 : 1;
    while (remaining > 0 && err == cudaSuccess)
    {
        for (int g = 0; g < n_groups && err == cudaSuccess; g++)
        {
            GroupRun& R = run[g];
            if (R.finished) continue;
            const WfGroup& G = groups[g];
            // has an earlier poll of this group's unfinished-pixel counter landed?
            if (R.poll_pending && cudaEventQuery(G.poll_event) == cudaSuccess)
            {
                R.poll_pending = false;
                if (*G.host_active == 0) { R.finished = true; remaining--; continue; }
                if (tail_ok && *G.host_active <= R.tail_below)
                {
                    // few pixels left: no more passes; one barrier-free launch finishes them, behind the passes already queued
                    WF_TRY(finish_group(g, R.P));
                    R.finished = true; remaining--;
                    continue;
                }
            }
            // bounded run-ahead: at most kRunAhead iterations queued behind an unanswered poll (a finished group would
            // otherwise leave a long train of empty launches behind)
            if (R.poll_pending && R.it - R.poll_it >= 8) continue;
            if (R.it >= max_iters)
            {
                // safety net: spp * (max_bounces + 1) iterations finish every pixel. Wait for the last poll; pixels still
                // unfinished now are a bug and are reported to the caller, never dropped silently.
                unsigned int left = 0;
                WF_TRY(cudaStreamSynchronize(G.stream));
                WF_TRY(cudaMemcpy(&left, &G.buf.counters[2], sizeof(left), cudaMemcpyDeviceToHost));
                unfinished += left;
                R.finished = true; remaining--;
                continue;
            }
            WfTimeline::Launch tll = { g, 0, 0, 0 };
            if (timing) cudaEventRecord(tev[0], G.stream);
            if (tln) { tll.e0 = tln->used; cudaEventRecord(tln->take(), G.stream); }
            trace_kernel<<<trace_grid, tb, 0, G.stream>>>(S, G.buf, R.parity);
            if (timing) cudaEventRecord(tev[1], G.stream);
            if (tln) { tll.e1 = tln->used; cudaEventRecord(tln->take(), G.stream); }
            R.parity ^= 1;
            wf_shade<<<(G.buf.n_slots + WF_SHADE_BLOCK - 1) / WF_SHADE_BLOCK, WF_SHADE_BLOCK, 0, G.stream>>>(S, R.P, G.buf, fb_in_rowmajor, out_tiles, R.parity);
            if (tln) { tll.e2 = tln->used; cudaEventRecord(tln->take(), G.stream); tln->launches.push_back(tll); }
            launches += 2;
            WF_TRY(cudaGetLastError());
            if (timing)
            {
                cudaEventRecord(tev[2], G.stream);
                WF_TRY(cudaEventSynchronize(tev[2]));
                float a = 0, b = 0;
                cudaEventElapsedTime(&a, tev[0], tev[1]); cudaEventElapsedTime(&b, tev[1], tev[2]);
                unsigned int nq[8] = {};
                WF_TRY(cudaMemcpy(nq, G.buf.counters, sizeof(nq), cudaMemcpyDeviceToHost));
                t_trace += a; t_shade += b; n_trace++; n_shade++;
                if (timing_env) fprintf(stderr, "wf g%d it %lld: trace %.3f ms  shade %.3f ms  active px %u  next queue %u\n", g, R.it, a, b, nq[2], nq[3 + R.parity]);
            }
            R.it++;
            if (!R.poll_pending && ((R.it & 3) == 0 || R.it >= max_iters))
            {
                WF_TRY(cudaMemcpyAsync(G.host_active, &G.buf.counters[2], sizeof(unsigned int), cudaMemcpyDeviceToHost, G.stream));
                WF_TRY(cudaEventRecord(G.poll_event, G.stream));
                if (err == cudaSuccess) { R.poll_pending = true; R.poll_it = R.it; }
            }
        }
    }
    // join (on every path, error or not): the caller's stream continues after every group that was forked
    for (int g = 0; g < n_groups; g++)
    {
        const WfGroup& G = groups[g];
        if (!run[g].forked) continue;
        const cudaError_t e1 = cudaEventRecord(G.join_event, G.stream);
        const cudaError_t e2 = e1 == cudaSuccess ? cudaStreamWaitEvent(stream, G.join_event, 0) : e1;
        if (err == cudaSuccess && e2 != cudaSuccess) err = e2;
    }
#undef WF_TRY
    if (timing)
    {
        if (timing_env) fprintf(stderr, "wf total: trace %.3f ms  shade %.3f ms  launches %d\n", t_trace, t_shade, launches);
        if (kernel_times4) { kernel_times4[0] = t_trace; kernel_times4[1] = t_shade; kernel_times4[2] = n_trace; kernel_times4[3] = n_shade; }
        for (int i = 0; i < 3; i++) cudaEventDestroy(tev[i]);
    }
    if (launches_out) *launches_out = launches;
    if (unfinished_out) *unfinished_out = unfinished;
    if (err != cudaSuccess) return err;
    return cudaGetLastError();
}

cudaEvent_t WfTimeline::take()
{
    if (used == pool.size())
    {
        cudaEvent_t e = nullptr;
        cudaEventCreate(&e);
        pool.push_back(e);
    }
    return pool[used++];
}

void WfTimeline::destroy()
{
    for (cudaEvent_t e : pool) if (e) cudaEventDestroy(e);
    pool.clear(); used = 0; launches.clear();
    if (origin) { cudaEventDestroy(origin); origin = nullptr; }
}

cudaError_t wavefront_timeline_summary(const WfTimeline& tl, WfTimelineSummary* out)
{
    WfTimelineSummary s = { 0.0, 0.0, 0.0, 0.0, 0, 0, 0 };
    for (const WfTimeline::Launch& L : tl.tails)
    {
        float a = 0.0f;
        const cudaError_t e = cudaEventElapsedTime(&a, tl.pool[L.e0], tl.pool[L.e1]);
        if (e != cudaSuccess) return e;
        s.tail_ms += a; s.tail_launches++;
    }
    std::vector<std::pair<float, float>> iv;
    iv.reserve(tl.launches.size());
    for (const WfTimeline::Launch& L : tl.launches)
    {
        float t0 = 0.0f, a = 0.0f, b = 0.0f;
        cudaError_t e = cudaEventElapsedTime(&t0, tl.origin, tl.pool[L.e0]);
        if (e == cudaSuccess) e = cudaEventElapsedTime(&a, tl.pool[L.e0], tl.pool[L.e1]);
        if (e == cudaSuccess) e = cudaEventElapsedTime(&b, tl.pool[L.e1], tl.pool[L.e2]);
        if (e != cudaSuccess) return e;
        s.trace_ms += a; s.shade_ms += b; s.trace_launches++; s.shade_launches++;
        iv.emplace_back(t0, t0 + a);
    }
    std::sort(iv.begin(), iv.end());
    float cur0 = 0.0f, cur1 = -1.0f;
    for (const auto& p : iv)
    {
        if (cur1 < cur0) { cur0 = p.first; cur1 = p.second; }
        else if (p.first <= cur1) cur1 = std::max(cur1, p.second);
        else { s.trace_union_ms += cur1 - cur0; cur0 = p.first; cur1 = p.second; }
    }
    if (cur1 >= cur0) s.trace_union_ms += cur1 - cur0;
    *out = s;
    return cudaSuccess;
}

// sums the groups' ray counters into *total (one tiny launch on the caller's stream, after the join)
__global__ void wf_sum_rays(const unsigned long long* a, const unsigned long long* b, const unsigned long long* c, const unsigned long long* d,
                            const unsigned long long* e2, const unsigned long long* f, const unsigned long long* g, const unsigned long long* h,
                            int n, unsigned long long* total)
{
    const unsigned long long* p[8] = { a, b, c, d, e2, f, g, h };
    unsigned long long s = 0;
    for (int i = 0; i < n; i++) s += *p[i];
    *total = s;
}

cudaError_t wavefront_sum_rays(const WfGroup* groups, int n_groups, unsigned long long* total, cudaStream_t stream)
{
    const unsigned long long* p[8];
    for (int i = 0; i < 8; i++) p[i] = groups[i < n_groups ? i : 0].buf.rays_total;
    wf_sum_rays<<<1, 1, 0, stream>>>(p[0], p[1], p[2], p[3], p[4], p[5], p[6], p[7], n_groups, total);
    return cudaGetLastError();
}

} // namespace b200rt
