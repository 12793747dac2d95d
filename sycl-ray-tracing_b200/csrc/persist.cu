// Persistent integrator (sm_100a; B200RT_INTEGRATOR_PERSISTENT): the wavefront integrator without its frame-wide barrier.
//
// The pass-synchronous integrator (wavefront.cu) advances EVERY pixel of a tile group by one shading step per launch pair, so a
// frame is a chain of up to spp * (max_bounces + 1) dependent passes, each as long as its slowest ray plus two launches —
// the bound of a rank that holds few pixels (one of 8 GPUs on a 1080p frame: 0.22 ms per iteration, DESIGN.md). Here every
// WARP is its own little wavefront machine: it owns K * 32 state slots, shades them (wf_shade_slot: the same device code,
// 27 of 32 lanes active), traces the rays they produced from a private queue with the same warp-cooperative traversal
// (coop_trace_queue), and repeats; a slot whose pixel finished pulls the next pixel from a global counter. Warps never
// wait for each other, there is one launch per frame, nothing is polled from the host, and a pixel's chain of iterations
// costs what ITS warp's rays cost. Same device functions on the same per-pixel RNG streams: the frame is bit-identical to
// the other integrators' and the ray count is the same.
#include <algorithm>
#include <cstdlib>

#include "wf_device.cuh"

namespace b200rt {

#ifndef PERSIST_MIN_BLOCKS
#define PERSIST_MIN_BLOCKS 5
#endif

template <int K>
__global__ void __launch_bounds__(32 * kCoopMaxWarps, PERSIST_MIN_BLOCKS)
pt_persist(SceneDev S, RenderParams P, WfBuffers B, unsigned int* next_pixel, int n_frame_slots, const float4* __restrict__ fb_in_rowmajor,
           float4* __restrict__ out_tiles)
{
    __shared__ CoopWarp s_warps[kCoopMaxWarps];
    __shared__ uint2 s_stack[kSharedStackDepth * 32 * kCoopMaxWarps];
    CoopWarp& W = s_warps[threadIdx.x >> 5];
    TravStack8Shared Kst;
    Kst.sh = s_stack + threadIdx.x; Kst.stride = 32 * kCoopMaxWarps;
    const unsigned int FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const unsigned int lanes_below = (1u << lane) - 1u;
    const int warp_global = blockIdx.x * kCoopMaxWarps + (threadIdx.x >> 5);
    const int base = warp_global * (K * 32);
    unsigned int* queue = B.queue + (size_t)warp_global * (K * 32 * 5);
    const bool no_paths = P.sample_end <= P.sample_begin || P.max_bounces <= 0;

    int st[K], px[K];
#pragma unroll
    for (int k = 0; k < K; k++) { st[k] = WF_DONE; px[k] = 0; }
    bool pool_empty = false;                    // warp-uniform
    unsigned long long rays = 0;

    for (;;)
    {
        unsigned int qn = 0;                    // warp-uniform: rays queued by this iteration's shading
#pragma unroll
        for (int k = 0; k < K; k++)
        {
            const int slot = base + k * 32 + lane;
            ShadeOut R;
            R.q_path = R.q0 = R.q1 = R.q2 = R.q3 = R.pixel_done = false; R.flags = st[k];
            if (!(st[k] & WF_DONE))
            {
                int x, y;
                wf_slot_pixel(P, px[k], x, y);
                R = wf_shade_slot(S, P, B, slot, st[k], x, y, (size_t)px[k], fb_in_rowmajor, out_tiles);
                st[k] = R.flags;
            }
            // slots without a pixel take the next ones of the frame (one atomic per warp and row)
            const bool need = (st[k] & WF_DONE) != 0 && !pool_empty;
            const unsigned int m = __ballot_sync(FULL, need);
            if (m)
            {
                const unsigned int cnt = __popc(m);
                unsigned int first = 0;
                if (lane == __ffs(m) - 1) first = atomicAdd(next_pixel, cnt);
                first = __shfl_sync(FULL, first, __ffs(m) - 1);
                const unsigned int mine = first + __popc(m & lanes_below);
                if (need && mine < (unsigned int)n_frame_slots)
                {
                    int x, y;
                    if (!wf_slot_pixel(P, (int)mine, x, y)) out_tiles[mine] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);     // tile padding outside the frame
                    else if (no_paths)
                    {
                        const float n = (float)P.spp;
                        out_tiles[mine] = pixel_output(P.flags, fb_in_rowmajor, (size_t)y * P.cam.w + x, CO(0.0f / n, 0.0f / n, 0.0f / n));
                    }
                    else
                    {
                        wf_begin_pixel(P, B, slot, x, y, (size_t)mine);
                        st[k] = WF_ALIVE; px[k] = (int)mine;
                        R.q_path = true;
                    }
                }
                if (first + cnt >= (unsigned int)n_frame_slots) pool_empty = true;
            }
            // this row's rays, grouped by kind like the pass-synchronous kernels' queue
            const unsigned int s3 = (unsigned int)slot << 3;
            const bool q[5] = { R.q_path, R.q0, R.q1, R.q2, R.q3 };
            const unsigned int tag[5] = { 4u, 0u, 1u, 2u, 3u };
#pragma unroll
            for (int j = 0; j < 5; j++)
            {
                const unsigned int mq = __ballot_sync(FULL, q[j]);
                if (q[j]) queue[qn + __popc(mq & lanes_below)] = s3 | tag[j];
                qn += __popc(mq);
            }
        }
        if (qn == 0)
        {
            // nothing to trace. Done only when no pixel is left to claim AND no slot has shading work left: a terminated path whose
            // side rays were all skipped produces no ray but still has to be shaded once more; claimed tile padding means claim again
            bool live = false;
#pragma unroll
            for (int k = 0; k < K; k++) live = live || !(st[k] & WF_DONE);
            if (pool_empty && !__any_sync(FULL, live)) break;
            continue;
        }
        rays += qn;
        __syncwarp();
        CoopQueuePrivate src;
        src.next = 0; src.end = qn;
        coop_trace_queue(S, B, queue, src, W, Kst);
        __syncwarp();
    }
    if (lane == 0 && rays) atomicAdd(B.rays_total, rays);
}

// ---- barrier-free tail of a pass-synchronous frame ------------------------------------------------------------------------------------
// A tile group's frame is a chain of up to spp * (max_bounces + 1) trace/shade passes, each as long as its slowest ray plus two
// launches (~0.19 ms when the passes are thin), although after the first 2 * spp passes only the pixels with long paths are
// still alive. Once few pixels are left, wavefront.cu stops launching passes: wf_compact_active lists the unfinished slots and
// ONE wf_tail launch finishes them. Every warp claims a few slots of that list and runs them to completion on its own — shade
// (wf_shade_slot), trace the rays from a private queue (coop_trace_queue), repeat — so a pixel's remaining chain costs what its
// own rays cost, not what the slowest ray of the group costs. Same state (the group's WfBuffers, in place), same device
// functions: the frame stays bit-identical.
__global__ void __launch_bounds__(256) wf_compact_active(WfBuffers B, unsigned int* list, unsigned int* n_active)
{
    const int slot = blockIdx.x * blockDim.x + threadIdx.x;
    const bool alive = slot < B.n_slots && !(B.flags[slot] & WF_DONE);
    wf_enqueue(list, n_active, alive, (unsigned int)slot);
}

__global__ void __launch_bounds__(32 * kCoopMaxWarps, PERSIST_MIN_BLOCKS)
wf_tail(SceneDev S, RenderParams P, WfBuffers B, const unsigned int* list, const unsigned int* n_active_ptr, unsigned int* claim_counter,
        unsigned int* queue_mem, const float4* __restrict__ fb_in_rowmajor, float4* __restrict__ out_tiles)
{
    __shared__ CoopWarp s_warps[kCoopMaxWarps];
    __shared__ uint2 s_stack[kSharedStackDepth * 32 * kCoopMaxWarps];
    CoopWarp& W = s_warps[threadIdx.x >> 5];
    TravStack8Shared Kst;
    Kst.sh = s_stack + threadIdx.x; Kst.stride = 32 * kCoopMaxWarps;
    const unsigned int FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const unsigned int lanes_below = (1u << lane) - 1u;
    const unsigned int total_warps = gridDim.x * kCoopMaxWarps;
    const unsigned int warp_global = blockIdx.x * kCoopMaxWarps + (threadIdx.x >> 5);
    unsigned int* queue = queue_mem + (size_t)warp_global * 160;
    const unsigned int n_active = *n_active_ptr;
    const int n = B.n_slots;
    // slots per claim: the whole list spread over the grid's warps, so that an almost empty machine gives every ray a lane of its own
    const unsigned int spc = min(32u, max(4u, (n_active + total_warps - 1) / total_warps));
    unsigned long long rays = 0;
    unsigned int finished_pixels = 0;

    for (;;)
    {
        unsigned int first = 0;
        if (lane == 0) first = atomicAdd(claim_counter, spc);
        first = __shfl_sync(FULL, first, 0);
        if (first >= n_active) break;
        const bool mine = (unsigned int)lane < spc && first + lane < n_active;
        const int slot = mine ? (int)list[first + lane] : 0;
        int st = mine ? B.flags[slot] : WF_DONE;
        int x = 0, y = 0;
        if (mine) wf_slot_pixel(P, slot, x, y);
        bool first_iteration = true;
        for (;;)
        {
            ShadeOut R;
            R.q_path = R.q0 = R.q1 = R.q2 = R.q3 = R.pixel_done = false; R.flags = st;
            if (!(st & WF_DONE))
            {
                if (first_iteration)
                {
                    // the rays the last shading pass left for a trace pass that is not going to run: rebuilt from the slot's state
                    if (st & WF_PENDING)
                    {
                        R.q0 = __float_as_int(B.ray_d[(size_t)0 * n + slot].w) != SIDE_NONE;
                        R.q1 = __float_as_int(B.ray_d[(size_t)1 * n + slot].w) != SIDE_NONE;
                        R.q2 = __float_as_int(B.ray_d[(size_t)2 * n + slot].w) != SIDE_NONE;
                        R.q3 = __float_as_int(B.ray_d[(size_t)3 * n + slot].w) != SIDE_NONE;
                    }
                    R.q_path = (st & WF_ALIVE) != 0;
                }
                else
                {
                    R = wf_shade_slot(S, P, B, slot, st, x, y, wf_out_index(B, slot), fb_in_rowmajor, out_tiles);
                    st = R.flags;
                    if (R.pixel_done) finished_pixels++;
                }
            }
            first_iteration = false;
            unsigned int qn = 0;
            const unsigned int s3 = (unsigned int)slot << 3;
            const bool q[5] = { R.q_path, R.q0, R.q1, R.q2, R.q3 };
            const unsigned int tag[5] = { 4u, 0u, 1u, 2u, 3u };
#pragma unroll
            for (int j = 0; j < 5; j++)
            {
                const unsigned int mq = __ballot_sync(FULL, q[j]);
                if (q[j]) queue[qn + __popc(mq & lanes_below)] = s3 | tag[j];
                qn += __popc(mq);
            }
            if (qn == 0)
            {
                // nothing to trace: either every slot is finished, or some slot has shading work that needs no ray (a terminated path
                // whose side rays were all skipped): shade again until rays or the end come out
                if (!__any_sync(FULL, !(st & WF_DONE))) break;
                continue;
            }
            rays += qn;
            __syncwarp();
            CoopQueuePrivate src;
            src.next = 0; src.end = qn;
            coop_trace_queue(S, B, queue, src, W, Kst);
            __syncwarp();
        }
    }
    for (int o = 16; o > 0; o >>= 1) finished_pixels += __shfl_down_sync(FULL, finished_pixels, o);
    if (lane == 0)
    {
        if (rays) atomicAdd(B.rays_total, rays);
        if (finished_pixels) atomicSub(&B.counters[2], finished_pixels);
    }
}

// B.queue is free once the passes have stopped: its first n_slots words hold the list of unfinished slots, the rest the warps'
// private ray queues (160 entries each). counters[6] = list length, counters[7] = claim counter (the pass kernels are done with both).
cudaError_t launch_wavefront_tail(const SceneDev& S, const RenderParams& P, const WfBuffers& B, int max_ctas, const float4* fb_in_rowmajor,
                                  float4* out_tiles, cudaStream_t stream)
{
    if (B.n_slots <= 0) return cudaSuccess;
    cudaError_t e;
    if ((e = cudaMemsetAsync(B.counters + 6, 0, 2 * sizeof(unsigned int), stream)) != cudaSuccess) return e;
    wf_compact_active<<<(B.n_slots + 255) / 256, 256, 0, stream>>>(B, B.queue, B.counters + 6);
    // private queues: 160 words per warp behind the list -> at most (4 * n_slots) / 160 warps
    const int max_warps = std::max(1, (int)(((size_t)4 * B.n_slots) / 160));
    int ctas = std::min(max_ctas, std::max(1, max_warps / kCoopMaxWarps));
    wf_tail<<<ctas, 32 * kCoopMaxWarps, 0, stream>>>(S, P, B, B.queue, B.counters + 6, B.counters + 7, B.queue + B.n_slots, fb_in_rowmajor, out_tiles);
    return cudaGetLastError();
}

int wavefront_tail_max_ctas()
{
    int per_sm = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, wf_tail, 32 * kCoopMaxWarps, 0);
    if (per_sm <= 0) per_sm = 1;
    return current_sm_count() * per_sm;
}

typedef void (*PersistKernel)(SceneDev, RenderParams, WfBuffers, unsigned int*, int, const float4*, float4*);

static PersistKernel persist_kernel(int k)
{
    return k == 1 ? pt_persist<1> : (k == 4 ? pt_persist<4> : pt_persist<2>);
}

int persistent_slots_per_lane()
{
    static const int k = []() { const char* e = getenv("B200RT_PERSIST_K"); const int v = e ? atoi(e) : 2; return (v == 1 || v == 4) ? v : 2; }();
    return k;
}

// CTAs of the persistent grid on the current device (a whole number per SM: every CTA is resident for the whole frame)
int persistent_grid()
{
    int per_sm = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, persist_kernel(persistent_slots_per_lane()), 32 * kCoopMaxWarps, 0);
    if (per_sm <= 0) per_sm = 1;
    static const int cap = []() { const char* e = getenv("B200RT_PERSIST_CTAS"); return e ? atoi(e) : 0; }();
    if (cap > 0 && cap < per_sm) per_sm = cap;
    return current_sm_count() * per_sm;
}

int persistent_slots(int grid) { return grid * kCoopMaxWarps * persistent_slots_per_lane() * 32; }

// B: state for persistent_slots(grid) slots (n_slots set accordingly), queue of 5 * n_slots entries, counters >= 1 word (the next-pixel
// counter), rays_total. The frame's pixels are this rank's tile-major slots [0, n_rank_tiles * 256); out_tiles is indexed by them.
cudaError_t run_persistent(const SceneDev& S, const RenderParams& P, const WfBuffers& B, int grid, const float4* fb_in_rowmajor,
                           float4* out_tiles, cudaStream_t stream)
{
    cudaError_t e;
    if ((e = cudaMemsetAsync(B.counters, 0, 8 * sizeof(unsigned int), stream)) != cudaSuccess) return e;
    if ((e = cudaMemsetAsync(B.rays_total, 0, sizeof(unsigned long long), stream)) != cudaSuccess) return e;
    const int n_frame_slots = P.n_rank_tiles * kTilePixels;
    if (n_frame_slots <= 0) return cudaSuccess;
    // no more warps than there are 32-pixel patches to start with
    const int warps_needed = (n_frame_slots + 31) / 32;
    const int ctas = std::min(grid, (warps_needed + kCoopMaxWarps - 1) / kCoopMaxWarps);
    persist_kernel(persistent_slots_per_lane())<<<ctas, 32 * kCoopMaxWarps, 0, stream>>>(S, P, B, B.counters, n_frame_slots, fb_in_rowmajor, out_tiles);
    return cudaGetLastError();
}

} // namespace b200rt
