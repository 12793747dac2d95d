// Device pieces shared by the pass-synchronous wavefront kernels (wavefront.cu) and the persistent integrator (persist.cu):
// the per-slot shading step (one surface interaction of render_kernel.cpp:96-162 per call) and the warp-cooperative
// closest / any-hit traversal of a queue of rays over the 8-ary BVH. Compiled with -fmad=false (see pt_device.cuh).
#pragma once
#include "kernels.h"
#include "pt_device.cuh"

namespace b200rt {

enum { WF_ALIVE = 1, WF_PENDING = 2, WF_TERMINATED = 4, WF_DONE = 8 };

// Loads of per-slot integrator state (WfBuffers) go to L2 (ld.global.cg), not through L1: a kernel reads each state word of a
// slot once per launch (DESIGN.md §2), so caching it in L1 would buy no reuse.
template <typename T>
__device__ __forceinline__ T wf_ld(const T* p) { return __ldcg(p); }

// appends `entry` for every lane with `pred` to queue[*counter ...] (one atomic per warp)
__device__ __forceinline__ void wf_enqueue(unsigned int* queue, unsigned int* counter, bool pred, unsigned int entry)
{
    const unsigned int mask = __ballot_sync(0xffffffffu, pred);
    if (!mask) return;
    const int lane = threadIdx.x & 31;
    const int leader = __ffs(mask) - 1;
    unsigned int base = 0;
    if (lane == leader) base = atomicAdd(counter, (unsigned int)__popc(mask));
    base = __shfl_sync(0xffffffffu, base, leader);
    if (pred) queue[base + __popc(mask & ((1u << lane) - 1u))] = entry;
}

// As wf_enqueue for up to five entries per lane with ONE reservation per warp (the shade kernels: path ray + four side rays):
// the warp's entries are laid out kind-major — all lanes' entry 0, then all lanes' entry 1, ... — so 32 neighbouring pixels' rays
// of one kind still sit side by side, and the warp waits for one returned atomic instead of five.
__device__ __forceinline__ void wf_enqueue5(unsigned int* queue, unsigned int* counter, const bool q[5], const unsigned int entry[5])
{
    const int lane = threadIdx.x & 31;
    const unsigned int below = (1u << lane) - 1u;
    unsigned int m[5], total = 0u;
#pragma unroll
    for (int k = 0; k < 5; k++) { m[k] = __ballot_sync(0xffffffffu, q[k]); total += __popc(m[k]); }
    if (!total) return;
    unsigned int base = 0;
    if (lane == 0) base = atomicAdd(counter, total);
    base = __shfl_sync(0xffffffffu, base, 0);
#pragma unroll
    for (int k = 0; k < 5; k++)
    {
        if (q[k]) queue[base + __popc(m[k] & below)] = entry[k];
        base += __popc(m[k]);
    }
}

__device__ __forceinline__ void wf_store_ray(const WfBuffers& B, int k, int slot, v3 o, v3 d, float tmax, int kind)
{
    const size_t i = (size_t)k * B.n_slots + slot;
    B.ray_o[i] = make_float4(o.x, o.y, o.z, tmax);
    B.ray_d[i] = make_float4(d.x, d.y, d.z, __int_as_float(kind));
}

__device__ __forceinline__ void wf_start_sample(const RenderParams& P, const WfBuffers& B, int slot, int x, int y, uint32_t& rng)
{
    const float xj = ((float)x + 0.5f) + xs_float(rng) - 1.0f;      // :88-89
    const float yj = ((float)y + 0.5f) + xs_float(rng) - 1.0f;
    v3 o, d;
    camera_ray(P.cam, xj, yj, o, d);
    wf_store_ray(B, 4, slot, o, d, 0.0f, SIDE_CLOSEST_LIGHT);
}

// where slot `slot` of a tile group writes its pixel: group g of G owns every G-th tile of the rank's tile-major buffer
__device__ __forceinline__ size_t wf_out_index(const WfBuffers& B, int slot)
{
    return ((size_t)(slot >> 8) * B.tile_stride + B.tile_offset) * kTilePixels + (slot & 255);
}

// pixel index of this rank's tile-major buffer (8x4 patches inside 16x16 tiles) -> pixel; false outside the frame
__device__ __forceinline__ bool wf_slot_pixel(const RenderParams& P, int slot, int& x, int& y)
{
    const int unit = slot >> 5, lane = slot & 31;
    const int k = unit >> 3, sub = unit & 7;
    int tx, ty;
    tile_xy(P.rank + k * P.world, P.tiles_x, P.tile_skew, tx, ty);
    x = tx * kTileDim + (sub & 1) * kPatchW + (lane & 7);
    y = ty * kTileDim + (sub >> 1) * kPatchH + (lane >> 3);
    return x < P.cam.w && y < P.cam.h;
}

// normal of an analytic sphere hit (Sphere::intersect, sphere.h:47-49), recomputed from the stored hit distance
__device__ __forceinline__ v3 wf_sphere_normal(const SceneDev& S, int prim, v3 p)
{
    for (int i = 0; i < S.n_spheres; i++)
    {
        const SphereDev s = S.spheres[i];
        if (s.prim == prim) return normalize(p - V(s.cx, s.cy, s.cz));
    }
    return V(0.0f, 0.0f, 0.0f);
}

// starts pixel (x, y) in state slot `slot`: RNG seed + warm-up (:77-82) — or, when a progressive accumulation continues, the
// generator state and radiance sum the pixel's previous samples left in acc_rng / acc_sum[out_index] — and the first camera
// ray into ray slot 4
__device__ __forceinline__ void wf_begin_pixel(const RenderParams& P, const WfBuffers& B, int slot, int x, int y, size_t out_index)
{
    const bool resume = P.acc_rng != nullptr && P.sample_begin > 0;
    uint32_t rng = resume ? P.acc_rng[out_index] : pixel_rng(x, y, P.spp);
    wf_start_sample(P, B, slot, x, y, rng);
    B.rng[slot] = rng;
    B.sample[slot] = P.sample_begin;
    B.bounce[slot] = 0;
    B.final_c[slot] = resume ? P.acc_sum[out_index] : make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    B.sample_c[slot] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    B.thr[slot] = make_float4(1.0f, 1.0f, 1.0f, 0.0f);
    B.flags[slot] = WF_ALIVE;
}

// what one shading step of a slot produced: which of its ray slots (0..3 side rays, 4 path ray) hold a ray to trace now
struct ShadeOut { bool q_path, q0, q1, q2, q3, pixel_done; int flags; };

// One shading step of state slot `slot`, whose pixel is (x, y) and whose result goes to out_tiles[out_index]:
//   A. resolve the side rays of the previous surface interaction (sample_color += (light + env) * throughput, :128)
//   B. consume the path ray's closest hit: miss -> sky (camera rays only, :146-159) and finish the sample; hit -> material
//      fetch, the four side rays of sample_light_sources / sample_environment_map with their MIS weights, the continuation
//      sample, the termination tests (:130-135)
//   C. finish the sample: the pixel's next sample (path regeneration) or the pixel itself
// The per-pixel RNG stream is consumed in exactly the reference's order.
__device__ __forceinline__ ShadeOut wf_shade_slot(const SceneDev& S, const RenderParams& P, const WfBuffers& B, int slot, int flags_in, int x, int y,
                                                  size_t out_index, const float4* __restrict__ fb_in_rowmajor, float4* __restrict__ out_tiles)
{
    ShadeOut R;
    R.q_path = R.q0 = R.q1 = R.q2 = R.q3 = R.pixel_done = false;
    R.flags = flags_in;
    const int n = B.n_slots;
    uint32_t rng = wf_ld(B.rng + slot);
    int sample = wf_ld(B.sample + slot), bounce = wf_ld(B.bounce + slot);
    float4 t4 = wf_ld(B.thr + slot), s4 = wf_ld(B.sample_c + slot);
    col throughput = CO(t4.x, t4.y, t4.z), sample_color = CO(s4.x, s4.y, s4.z);
    int flags = flags_in;
    bool finish = false;
    const bool trace_light_brdf = S.any_emissive_material || !(P.flags & B200RT_FLAG_SKIP_DEAD_RAYS);

    // A. resolve the side rays of the previous surface interaction
    if (flags & WF_PENDING)
    {
        col c[4];
#pragma unroll
        for (int k = 0; k < 4; k++)
        {
            c[k] = CO(0.0f, 0.0f, 0.0f);
            const size_t i = (size_t)k * n + slot;
            const float4 rd4 = wf_ld(B.ray_d + i);
            const int kind = __float_as_int(rd4.w);
            if (kind == SIDE_NONE) continue;
            const float4 w4 = wf_ld(B.side_w + i);
            const float4 res = wf_ld(B.res + i);      // {t, primitive | occlusion flag, triangle slot, -}
            if (kind == SIDE_CLOSEST_LIGHT)
            {
                const float t = res.x;
                if (t > 0.0f)
                {
                    const float4 ro4 = wf_ld(B.ray_o + i);
                    SideRay sr;
                    sr.o = V(ro4.x, ro4.y, ro4.z); sr.d = V(rd4.x, rd4.y, rd4.z);
                    sr.weight = CO(w4.x, w4.y, w4.z); sr.pdf = w4.w; sr.kind = kind; sr.tmax = 0.0f;
                    Hit h;
                    h.t = t; h.prim = __float_as_int(res.y); h.slot = __float_as_int(res.z); h.u = h.v = -1.0f;
                    if (h.slot < 0) h.sphere_n = wf_sphere_normal(S, h.prim, sr.o + t * sr.d);
                    c[k] = side_light_hit(S, sr, h);
                }
            }
            else if (__float_as_int(res.y) == 0) c[k] = CO(w4.x, w4.y, w4.z);      // unoccluded
        }
        sample_color = sample_color + ((c[0] + c[1]) + (c[3] + c[2])) * throughput;     // light = c0+c1 (:712), env = c3+c2 (:630), :128
        const float4 tn = wf_ld(B.thr_next + slot);
        throughput = CO(tn.x, tn.y, tn.z);
        flags &= ~WF_PENDING;
        if (flags & WF_TERMINATED) finish = true;
    }

    // B. consume the path ray
    if (!finish && (flags & WF_ALIVE))
    {
        const size_t i = (size_t)4 * n + slot;
        const float4 ro4 = wf_ld(B.ray_o + i), rd4 = wf_ld(B.ray_d + i);
        const v3 ro = V(ro4.x, ro4.y, ro4.z), rd = V(rd4.x, rd4.y, rd4.z);
        const float4 res = wf_ld(B.res + i);
        const float t = res.x;
        if (!(t > 0.0f))
        {
            if (bounce == 0 && P.max_bounces >= 2)                           // :146-159
                sample_color = sample_color + env_from_direction(S, rd) * throughput;
            finish = true;
        }
        else
        {
            Hit h;
            h.t = t; h.prim = __float_as_int(res.y); h.slot = __float_as_int(res.z); h.u = h.v = -1.0f;
            Surface sf;
            sf.p = ro + t * rd;
            if (h.slot >= 0)
            {
                const float4 ve1 = __ldg(S.tris + 3 * (size_t)h.slot + 1), ve2 = __ldg(S.tris + 3 * (size_t)h.slot + 2);
                sf.n = normalize(cross(V(ve1.x, ve1.y, ve1.z), V(ve2.x, ve2.y, ve2.z)));
            }
            else sf.n = wf_sphere_normal(S, h.prim, sf.p);
            sf.view = -rd;
            sf.m = S.mats[__ldg(S.mat_idx + h.prim)];                        // :107-108
            SideRay sr;
            sr.o = sr.d = V(0.0f, 0.0f, 0.0f); sr.tmax = 0.0f; sr.pdf = 0.0f; sr.weight = CO(0.0f, 0.0f, 0.0f);
            side_light_sample(S, sf, rng, sr);
            wf_store_ray(B, 0, slot, sr.o, sr.d, sr.tmax, sr.kind);
            if (sr.kind != SIDE_NONE) { B.side_w[(size_t)0 * n + slot] = make_float4(sr.weight.r, sr.weight.g, sr.weight.b, 0.0f); R.q0 = true; }
            side_light_brdf(S, sf, rng, sr);
            if (sr.kind != SIDE_NONE && !trace_light_brdf) sr.kind = SIDE_NONE;
            wf_store_ray(B, 1, slot, sr.o, sr.d, 0.0f, sr.kind);
            if (sr.kind != SIDE_NONE) { B.side_w[(size_t)1 * n + slot] = make_float4(sr.weight.r, sr.weight.g, sr.weight.b, sr.pdf); R.q1 = true; }
            side_env_sample(S, sf, rng, sr);
            wf_store_ray(B, 2, slot, sr.o, sr.d, 0.0f, sr.kind);
            if (sr.kind != SIDE_NONE) { B.side_w[(size_t)2 * n + slot] = make_float4(sr.weight.r, sr.weight.g, sr.weight.b, 0.0f); R.q2 = true; }
            side_env_brdf(S, sf, rng, sr);
            wf_store_ray(B, 3, slot, sr.o, sr.d, 0.0f, sr.kind);
            if (sr.kind != SIDE_NONE) { B.side_w[(size_t)3 * n + slot] = make_float4(sr.weight.r, sr.weight.g, sr.weight.b, 0.0f); R.q3 = true; }

            float bpdf;
            v3 ndir = V(0.0f, 0.0f, 0.0f);
            const col brdf = ct_sample(sf.m, sf.view, sf.n, ndir, bpdf, rng);        // :123
            if (bounce == 0) sample_color = sample_color + CO(sf.m.er, sf.m.eg, sf.m.eb);
            flags = WF_PENDING;
            col tnext = throughput;
            if (is_black(brdf) || bpdf < 1.0e-8f || isinf(bpdf)) flags |= WF_TERMINATED;     // :130-135
            else
            {
                tnext = throughput * ((brdf * smax(0.0f, dot(ndir, sf.n))) / bpdf);       // :137
                bounce++;
                if (bounce >= P.max_bounces) flags |= WF_TERMINATED;
                else
                {
                    wf_store_ray(B, 4, slot, sf.p + 1.0e-4f * sf.n, ndir, 0.0f, SIDE_CLOSEST_LIGHT);
                    flags |= WF_ALIVE;
                    R.q_path = true;
                }
            }
            B.thr_next[slot] = make_float4(tnext.r, tnext.g, tnext.b, 0.0f);
        }
    }

    // C. finish the sample: next sample of this pixel, or the pixel itself
    if (finish)
    {
        float4 f4 = wf_ld(B.final_c + slot);
        col final_color = CO(f4.x, f4.y, f4.z) + sample_color;
        sample++;
        if (sample < P.sample_end)
        {
            B.final_c[slot] = make_float4(final_color.r, final_color.g, final_color.b, 0.0f);
            wf_start_sample(P, B, slot, x, y, rng);
            throughput = CO(1.0f, 1.0f, 1.0f);
            sample_color = CO(0.0f, 0.0f, 0.0f);
            bounce = 0;
            flags = WF_ALIVE;
            R.q_path = true;
        }
        else
        {
            if (P.acc_rng) { P.acc_rng[out_index] = rng; P.acc_sum[out_index] = make_float4(final_color.r, final_color.g, final_color.b, 0.0f); }
            const float nspp = (float)P.sample_end;          // == spp for a one-shot frame and for the last chunk of an accumulation
            const col mean = CO(final_color.r / nspp, final_color.g / nspp, final_color.b / nspp);
            out_tiles[out_index] = pixel_output(P.flags, fb_in_rowmajor, (size_t)y * P.cam.w + x, mean);
            flags = WF_DONE;
            R.pixel_done = true;
        }
    }
    B.rng[slot] = rng;
    B.sample[slot] = sample;
    B.bounce[slot] = bounce;
    B.thr[slot] = make_float4(throughput.r, throughput.g, throughput.b, 0.0f);
    B.sample_c[slot] = make_float4(sample_color.r, sample_color.g, sample_color.b, 0.0f);
    B.flags[slot] = flags;
    R.flags = flags;
    return R;
}

// result of one queue entry: one 16-byte record {t or -1, primitive (closest hit) | occlusion flag (any-hit / shadow rays),
// triangle slot, 0}, written with a single 16-byte store.
__device__ __forceinline__ void wf_store_result(const WfBuffers& B, size_t r, int mode, bool found, const Hit& h)
{
    float4 v;
    if (mode == TRACE_CLOSEST) v = make_float4(found ? h.t : -1.0f, __int_as_float(h.prim), __int_as_float(h.slot), 0.0f);
    else v = make_float4(0.0f, __int_as_float(found ? 1 : 0), 0.0f, 0.0f);
    B.res[r] = v;
}

// ---- warp-cooperative traversal of a ray queue over the 8-ary BVH -----------------------------------------------------------------
// Every lane owns one traversal state and is refilled from the queue as soon as enough lanes are idle (persistent threads, per
// lane). A lane never tests its own triangles. After a node step it leaves ONE descriptor {owner lane | first triangle slot,
// hit bits, valid24} of the node's hit leaf children in a per-warp shared-memory ring (one ballot + one store for the whole
// warp) and goes straight on with its next node. When the ring holds kCoopDrainTris triangles, the warp expands the front
// descriptors into exactly that many (owner, triangle) pairs — a descriptor is split when it straddles the limit — and all 32
// lanes run Moller-Trumbore (triangle.h:16-60) on one pair each per batch, folding hits into the owner's 64-bit key
// (t bits << 32 | primitive index) with a shared-memory atomicMin: exactly the closest-hit rule of every other kernel here
// (smaller t, ties to the lower original index), in whatever order the tests run. Owners pick up their new t_best after each
// drain; a ray is finished when it has no node work and no descriptor left in the ring.
// (Round 1 appended every (owner, triangle) pair separately in a per-lane loop: 13.5 % of the kernel's instructions at 4.4
// active lanes, profiles/r1b_blocks_wf_trace_coop_c3.txt.)
#ifndef WF_WARP_BLOCK
#define WF_WARP_BLOCK 64
#endif
#ifndef WF_REFILL
#define WF_REFILL 8
#endif
#ifndef WF_COOP_DRAIN_TRIS
#define WF_COOP_DRAIN_TRIS 64
#endif
#ifndef WF_COOP_RING
#define WF_COOP_RING 64
#endif
constexpr int kWarpBlock = WF_WARP_BLOCK;
constexpr int kRefillThreshold = WF_REFILL;
constexpr int kCoopDrainTris = WF_COOP_DRAIN_TRIS;      // 32 or 64: pairs tested per drain
constexpr int kCoopRing = WF_COOP_RING;                 // descriptors per warp (power of two, >= 64: a node step appends up to 32 and
                                                        // a drain leaves at most 32 behind)
constexpr int kCoopWork = 96;                           // expanded pairs per drain when flushing (>= kCoopDrainTris, multiple of 32)
constexpr int kCoopMaxWarps = 4;                        // the kernels are launched with 128-thread CTAs
constexpr unsigned long long kNoHit = 0xffffffffffffffffull;
static_assert((kCoopRing & (kCoopRing - 1)) == 0 && kCoopRing >= 64, "ring size");
static_assert(kCoopDrainTris == 32 || kCoopDrainTris == 64, "drain size");

struct CoopWarp
{
    float4 ro[32], rd[32];              // per lane: origin + tmax, direction + trace mode
    unsigned long long best[32];        // per lane: (t bits << 32) | primitive index of the best accepted hit
    unsigned int dx[kCoopRing];         // descriptor ring: (owner lane << 27) | first triangle slot of the node
    unsigned int dy[kCoopRing];         //                  hit bits in valid24 positions (what is left of them after a split)
    unsigned int dz[kCoopRing];         //                  valid24 of the node
    unsigned int work[kCoopWork];       // expanded (owner lane << 27) | triangle slot pairs of the current drain
    unsigned int pend[32];              // per lane: descriptors of this lane still in the ring
};

// One drain. limit = number of pairs to expand and test now (<= kCoopWork, <= qtris). Warp-uniform: head, dcount, qtris.
__device__ __forceinline__ void coop_drain(const SceneDev& S, CoopWarp& W, const int lane, unsigned int& head, unsigned int& dcount,
                                           unsigned int& qtris, const unsigned int limit)
{
    const unsigned int FULL = 0xffffffffu;
    const unsigned int nd = min(32u, dcount);
    const unsigned int di = (head + (unsigned int)lane) & (kCoopRing - 1);
    unsigned int x = 0, bits = 0, valid = 0;
    if ((unsigned int)lane < nd) { x = W.dx[di]; bits = W.dy[di]; valid = W.dz[di]; }
    const unsigned int cnt = __popc(bits);
    unsigned int incl = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1)
    {
        const unsigned int up = __shfl_up_sync(FULL, incl, o);
        if (lane >= o) incl += up;
    }
    const unsigned int lim = min(limit, __shfl_sync(FULL, incl, 31));      // the first nd descriptors may hold fewer than `limit` triangles
    unsigned int pos = incl - cnt;
    // expand: the usual descriptor holds 1-3 triangles (three straight-line rounds); the rest loops
    const unsigned int owner_bits = x & 0xf8000000u, base = x & 0x07ffffffu;
#pragma unroll
    for (int r = 0; r < 3; r++)
    {
        if (bits && pos < lim)
        {
            const int b = __ffs((int)bits) - 1;
            bits &= bits - 1u;
            W.work[pos++] = owner_bits | (base + __popc(valid & ((1u << b) - 1u)));
        }
    }
    while (bits && pos < lim)
    {
        const int b = __ffs((int)bits) - 1;
        bits &= bits - 1u;
        W.work[pos++] = owner_bits | (base + __popc(valid & ((1u << b) - 1u)));
    }
    // descriptors that were expanded completely leave the ring; the one that straddles the limit keeps its remaining bits
    const bool touched = (unsigned int)lane < nd && incl - cnt < lim;
    const bool whole = touched && bits == 0u;
    if (touched && !whole) W.dy[di] = bits;
    const unsigned int n_whole = __popc(__ballot_sync(FULL, whole));
    __syncwarp();
    for (unsigned int base_i = 0; base_i < lim; base_i += 32u)
    {
        const unsigned int i = base_i + (unsigned int)lane;
        if (i < lim)
        {
            const unsigned int e = W.work[i];
            const unsigned int owner = e >> 27, slot = e & 0x07ffffffu;
            const float4 ro4 = W.ro[owner], rd4 = W.rd[owner];
            const float4* tp = S.tris + 3 * (size_t)slot;
            const float4 va = __ldg(tp), ve1 = __ldg(tp + 1), ve2 = __ldg(tp + 2);
            float t, u, v;
            if (tri_test(va, ve1, ve2, V(ro4.x, ro4.y, ro4.z), V(rd4.x, rd4.y, rd4.z), t, u, v))
            {
                const int mode = __float_as_int(rd4.w);
                if (mode != TRACE_SHADOW || t + 1.0e-4f < ro4.w)
                {
                    const unsigned long long key = ((unsigned long long)__float_as_uint(t) << 32) | (unsigned int)__float_as_int(va.w);
                    if (key < W.best[owner]) atomicMin(&W.best[owner], key);
                }
            }
        }
    }
    __syncwarp();
    if (whole) atomicSub(&W.pend[x >> 27], 1u);
    __syncwarp();
    head = (head + n_whole) & (kCoopRing - 1);
    dcount -= n_whole;
    qtris -= lim;
}

// Where a warp gets its rays from: blocks of a queue claimed with one atomic (the pass-synchronous kernels: every warp of
// the grid shares one queue) or a private range (the persistent integrator: a warp traces the rays its own slots produced).
struct CoopQueueShared
{
    static constexpr bool kCacheEntries = true;       // blocks of at most kWarpBlock entries: a claimed block's entries live in registers
    unsigned int* head; unsigned int n_rays, warp_block;
    __device__ __forceinline__ bool claim(int lane, unsigned int& blk_next, unsigned int& blk_end)
    {
        unsigned int b = 0;
        if (lane == 0) b = atomicAdd(head, warp_block);
        b = __shfl_sync(0xffffffffu, b, 0);
        if (b >= n_rays) return false;
        blk_next = b; blk_end = min(b + warp_block, n_rays);
        return true;
    }
};
struct CoopQueuePrivate
{
    static constexpr bool kCacheEntries = false;
    unsigned int next, end;
    __device__ __forceinline__ bool claim(int, unsigned int& blk_next, unsigned int& blk_end)
    {
        if (next >= end) return false;
        blk_next = next; blk_end = end; next = end;
        return true;
    }
};

// Traces every ray of the source's queue entries ((slot << 3) | k -> ray record k * n_slots + slot of B). All 32 lanes of the
// warp must call this together.
template <typename Source, typename Stack>
__device__ __forceinline__ void coop_trace_queue(const SceneDev& S, const WfBuffers& B, const unsigned int* queue, Source src,
                                                 CoopWarp& W, Stack& K)
{
    const unsigned int FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const unsigned int lanes_below = (1u << lane) - 1u;
    const int n = B.n_slots;
    const bool spheres = S.n_spheres != 0;

    Trav8 T;
    T.done = true; T.tg = make_uint2(0u, 0u);
    bool active = false;
    size_t r = 0;
    int mode = TRACE_CLOSEST;
    unsigned int blk_next = 0, blk_end = 0, blk_base = 0;      // warp-uniform: the warp's current block of queue entries
    unsigned int qe[kWarpBlock / 32 > 0 ? kWarpBlock / 32 : 1] = {};   // kCacheEntries: this lane's share of the block's entries
    unsigned int head = 0, dcount = 0, qtris = 0;              // warp-uniform: descriptor ring
    bool exhausted = false;                                    // warp-uniform
    W.pend[lane] = 0u;
    __syncwarp();

    for (;;)
    {
        // (1) refill idle lanes from the warp's block of the ray queue
        unsigned int idle = __ballot_sync(FULL, !active);
        if (idle && !exhausted && (idle == FULL || __popc(idle) >= kRefillThreshold))
        {
            if (blk_next >= blk_end)
            {
                if (!src.claim(lane, blk_next, blk_end)) exhausted = true;
                else if constexpr (Source::kCacheEntries)
                {
                    // the whole block's entries at once (lane l holds entries l, 32 + l, ...): the refills below then cost one
                    // dependent round trip (the ray record) instead of two
                    blk_base = blk_next;
#pragma unroll
                    for (int j = 0; j < kWarpBlock / 32; j++)
                    {
                        const unsigned int qi = blk_base + 32u * j + (unsigned int)lane;
                        qe[j] = qi < blk_end ? queue[qi] : 0u;
                    }
#ifndef B200RT_NO_RAY_PREFETCH
                    // ... and the ray records those entries name start moving towards L1 now (a pass kernel reads each of them
                    // exactly once, through L1: see the load below)
#pragma unroll
                    for (int j = 0; j < kWarpBlock / 32; j++)
                        if (blk_base + 32u * j + (unsigned int)lane < blk_end)
                        {
                            const size_t pr = (size_t)(qe[j] & 7u) * n + (qe[j] >> 3);
                            asm volatile("prefetch.global.L1 [%0];" ::"l"(B.ray_o + pr));
                            asm volatile("prefetch.global.L1 [%0];" ::"l"(B.ray_d + pr));
                        }
#endif
                }
            }
            if (blk_next < blk_end)
            {
                const unsigned int idx = blk_next + __popc(idle & lanes_below);
                unsigned int e = 0u;
                if constexpr (Source::kCacheEntries)
                {
                    const unsigned int rel = idx - blk_base;
#pragma unroll
                    for (int j = 0; j < kWarpBlock / 32; j++)
                    {
                        const unsigned int v = __shfl_sync(FULL, qe[j], (int)(rel & 31u));
                        if ((rel >> 5) == (unsigned int)j) e = v;
                    }
                }
                if (!active && idx < blk_end)
                {
                    if constexpr (!Source::kCacheEntries) e = queue[idx];
                    const int slot = (int)(e >> 3), k = (int)(e & 7u);
                    r = (size_t)k * n + slot;
                    // (kCacheEntries = a pass kernel: the records were written by the previous launch, plain loads find the prefetched lines)
                    const float4 ro4 = Source::kCacheEntries ? B.ray_o[r] : wf_ld(B.ray_o + r), rd4 = Source::kCacheEntries ? B.ray_d[r] : wf_ld(B.ray_d + r);
                    const int kind = __float_as_int(rd4.w);
                    mode = kind == SIDE_SHADOW ? TRACE_SHADOW : (kind == SIDE_CLOSEST_LIGHT ? TRACE_CLOSEST : TRACE_ANY);
                    const int tmode = spheres ? TRACE_CLOSEST : mode;
                    trav8_init(T, V(ro4.x, ro4.y, ro4.z), V(rd4.x, rd4.y, rd4.z), ro4.w, tmode);
                    W.ro[lane] = ro4;
                    W.rd[lane] = make_float4(rd4.x, rd4.y, rd4.z, __int_as_float(tmode));
                    W.best[lane] = kNoHit;
                    active = true;
                }
                blk_next = min(blk_next + (unsigned int)__popc(idle), blk_end);
            }
            __syncwarp();
        }
        if (!__any_sync(FULL, active))
        {
            if (exhausted) break;
            continue;
        }
        // (2) one node step for every lane that has one
        if (active && !T.done)
        {
            trav8_node(S, T, K);
            // the next node group can be fetched from the stack right away (its load overlaps the housekeeping below);
            // the pending triangle group lives in T.tg / T.tvalid, which the pop does not touch
            if (!T.done && !(T.ng.y & 0xff000000u)) trav8_pop(T, K);
        }
        // (3) hit leaf children -> one descriptor per lane in the warp's ring; the lane moves on
        {
            const bool has = active && T.tg.y != 0u;
            const unsigned int m = __ballot_sync(FULL, has);
            if (m)
            {
                if (has)
                {
                    const unsigned int di = (head + dcount + __popc(m & lanes_below)) & (kCoopRing - 1);
                    W.dx[di] = ((unsigned int)lane << 27) | T.tg.x;
                    W.dy[di] = T.tg.y;
                    W.dz[di] = T.tvalid;
                    W.pend[lane] += 1u;
                }
                qtris += __reduce_add_sync(FULL, has ? (unsigned int)__popc(T.tg.y) : 0u);
                dcount += __popc(m);
                T.tg.y = 0u;
                __syncwarp();
            }
        }
        // (4) test queued triangles: kCoopDrainTris at a time; everything when no lane has node work left or enough lanes wait
        const unsigned int m_node = __ballot_sync(FULL, active && !T.done);
        const unsigned int m_wait = __ballot_sync(FULL, active && T.done && W.pend[lane] != 0u);
        const bool flush = !m_node || __popc(m_wait) >= kRefillThreshold;
        if (qtris >= (unsigned int)kCoopDrainTris || dcount > (unsigned int)(kCoopRing - 32) || (flush && qtris))
        {
            do
            {
                // whole batches while the ring holds enough; the ring must keep room for 32 new descriptors; a flush takes everything
                unsigned int limit = qtris >= (unsigned int)kCoopDrainTris ? (unsigned int)kCoopDrainTris : min(qtris, 32u);
                if (flush || dcount > (unsigned int)(kCoopRing - 32)) limit = min(qtris, (unsigned int)kCoopWork);
                coop_drain(S, W, lane, head, dcount, qtris, limit);
            } while (qtris >= (unsigned int)kCoopDrainTris || dcount > (unsigned int)(kCoopRing - 32) || (flush && qtris));
            if (active)
            {
                const unsigned long long key = W.best[lane];
                if (key != kNoHit)
                {
                    if (T.mode == TRACE_CLOSEST) T.tbest = __uint_as_float((unsigned int)(key >> 32));
                    else T.done = true;           // occlusion established; the lane only waits for its queued descriptors to leave
                }
            }
        }
        // (5) finished rays
        if (active && T.done && W.pend[lane] == 0u)
        {
            const unsigned long long key = W.best[lane];
            Hit h;
            bool found = key != kNoHit;
            h.t = found ? __uint_as_float((unsigned int)(key >> 32)) : -1.0f;
            h.prim = found ? (int)(unsigned int)key : -1;
            h.slot = (found && T.mode == TRACE_CLOSEST) ? __ldg(S.slot_of_prim + h.prim) : -1;
            h.u = h.v = -1.0f;
            if (spheres)
            {
                const float4 ro4 = W.ro[lane], rd4 = W.rd[lane];
                found = finish_with_spheres(S, V(ro4.x, ro4.y, ro4.z), V(rd4.x, rd4.y, rd4.z), ro4.w, mode, h);
            }
            active = false;
            wf_store_result(B, r, mode, found, h);
        }
    }
}

} // namespace b200rt
