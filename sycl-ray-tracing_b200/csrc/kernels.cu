// sm_100a kernels of the path: primary closest-hit (K1), megakernel integrator (K2), ray batches, untile (K4).
// Compiled with -fmad=false (see pt_device.cuh).
#include <algorithm>

#include "kernels.h"
#include "pt_device.cuh"

namespace b200rt {

// pixel <-> work-unit mapping: a frame is cut into 16x16 tiles owned round-robin by ranks; a tile is 8 warp patches of
// 8x4 pixels; one warp renders one patch so its 32 rays start as a compact screen-space bundle.
struct PixelSlot { int x, y; size_t out; bool inside; };

__device__ __forceinline__ PixelSlot unit_pixel(const RenderParams& P, int unit, int lane)
{
    const int k = unit >> 3, sub = unit & 7;
    int tx, ty;
    tile_xy(P.rank + k * P.world, P.tiles_x, P.tile_skew, tx, ty);
    PixelSlot s;
    s.x = tx * kTileDim + (sub & 1) * kPatchW + (lane & 7);
    s.y = ty * kTileDim + (sub >> 1) * kPatchH + (lane >> 3);
    s.out = (size_t)k * kTilePixels + sub * 32 + lane;
    s.inside = s.x < P.cam.w && s.y < P.cam.h;
    return s;
}

// ---- K2: megakernel. One lane = one pixel at a time; a pixel's samples and bounces run in that lane so the pixel's
// xorshift stream is consumed in the reference's order (render_kernel.cpp:75-181). Persistent warps: every lane is a
// small state machine with ONE trace site per loop iteration — camera rays, continuation rays and the four side rays
// of a surface interaction all go through the same traversal call, a finished sample starts the next one in the same
// iteration, and a lane that finishes its pixel immediately pulls the next pixel slot from a global counter. Nothing
// ever waits for the slowest path of a warp except at the very end of the frame.
struct LaneState
{
    // pixel
    int x, y; unsigned int slot; uint32_t rng; int sample; col final_color;
    // path
    v3 ro, rd; float tmax; int mode; int stage; int bounce;
    col throughput, sample_color, c0, c1, c2, c3;
    Surface sf; SideRay sr;
};

__device__ __forceinline__ void start_sample(const RenderParams& P, LaneState& L)
{
    const float xj = ((float)L.x + 0.5f) + xs_float(L.rng) - 1.0f;      // :88-89
    const float yj = ((float)L.y + 0.5f) + xs_float(L.rng) - 1.0f;
    camera_ray(P.cam, xj, yj, L.ro, L.rd);
    L.throughput = CO(1.0f, 1.0f, 1.0f);
    L.sample_color = CO(0.0f, 0.0f, 0.0f);
    L.bounce = 0; L.stage = 4; L.mode = TRACE_CLOSEST; L.tmax = 0.0f;
    L.sr.kind = SIDE_NONE;
}

// slot (tile-major index into this rank's tile buffer) -> pixel; consecutive slots are the lanes of one 8x4 patch
__device__ __forceinline__ bool slot_pixel(const RenderParams& P, unsigned int slot, int& x, int& y)
{
    if (P.rw > 0)
    {
        x = P.rx0 + (int)(slot % (unsigned int)P.rw);
        y = P.ry0 + (int)(slot / (unsigned int)P.rw);
        return x < P.cam.w && y < P.cam.h;
    }
    const PixelSlot ps = unit_pixel(P, (int)(slot >> 5), (int)(slot & 31u));
    x = ps.x; y = ps.y;
    return ps.inside;
}

template <int TL>
__global__ void __launch_bounds__(256) k_pathtrace_mega(SceneDev S, RenderParams P, const float4* __restrict__ fb_in_rowmajor,
                                                        float4* __restrict__ out_tiles, unsigned int* work_counter,
                                                        unsigned long long* ray_counter)
{
    const unsigned int FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const unsigned int n_slots = P.rw > 0 ? (unsigned int)(P.rw * P.rh) : (unsigned int)P.n_rank_tiles * kTilePixels;
    const bool trace_light_brdf = S.any_emissive_material || !(P.flags & B200RT_FLAG_SKIP_DEAD_RAYS);
    const bool no_paths = P.spp <= 0 || P.max_bounces <= 0;
    unsigned long long rays = 0;
    bool have_pixel = false, exhausted = false;
    LaneState L;

    for (;;)
    {
        // (1) idle lanes pull the next pixel slot
        while (!have_pixel && !exhausted)
        {
            const unsigned int slot = atomicAdd(work_counter, 1u);
            if (slot >= n_slots) { exhausted = true; break; }
            int x, y;
            if (!slot_pixel(P, slot, x, y)) { out_tiles[slot] = make_float4(0.0f, 0.0f, 0.0f, 0.0f); continue; }
            if (no_paths)
            {
                const float n = (float)P.spp;
                out_tiles[slot] = pixel_output(P.flags, fb_in_rowmajor, (size_t)y * P.cam.w + x, CO(0.0f / n, 0.0f / n, 0.0f / n));
                continue;
            }
            L.x = x; L.y = y; L.slot = slot;
            L.rng = pixel_rng(x, y, P.spp);
            L.sample = 0;
            L.final_color = CO(0.0f, 0.0f, 0.0f);
            start_sample(P, L);
            have_pixel = true;
        }
        if (__all_sync(FULL, !have_pixel)) break;
        if (!have_pixel) continue;

        // (2) the single trace site
        Hit h;
        const bool found = trace_ray<TL>(S, L.ro, L.rd, L.tmax, L.mode, h);
        rays++;

        // (3) consume the result
        bool sample_done = false;
        if (L.stage == 4)
        {
            if (!found)
            {
                // MISSED is handled one loop iteration later and only adds the sky when that iteration is bounce 1 (:146-159)
                if (L.bounce == 0 && P.max_bounces >= 2)
                    L.sample_color = L.sample_color + env_from_direction(S, L.rd) * L.throughput;
                sample_done = true;
            }
            else
            {
                hit_geometry(S, h, L.ro, L.rd, L.sf.p, L.sf.n);
                L.sf.view = -L.rd;
                L.sf.m = S.mats[__ldg(S.mat_idx + h.prim)];                      // :107-108
                L.c0 = L.c1 = L.c2 = L.c3 = CO(0.0f, 0.0f, 0.0f);
                L.stage = 0;
            }
        }
        else
        {
            col c = CO(0.0f, 0.0f, 0.0f);
            if (L.sr.kind == SIDE_CLOSEST_LIGHT) { if (found) c = side_light_hit(S, L.sr, h); }
            else if (!found) c = L.sr.weight;
            if (L.stage == 0) L.c0 = c; else if (L.stage == 1) L.c1 = c; else if (L.stage == 2) L.c2 = c; else L.c3 = c;
            L.stage++;
        }

        // (4) advance to the next ray this lane has to trace
        while (!sample_done)
        {
            if (L.stage < 4)
            {
                if (L.stage == 0) side_light_sample(S, L.sf, L.rng, L.sr);
                else if (L.stage == 1) side_light_brdf(S, L.sf, L.rng, L.sr);
                else if (L.stage == 2) side_env_sample(S, L.sf, L.rng, L.sr);
                else side_env_brdf(S, L.sf, L.rng, L.sr);
                const bool need = L.sr.kind != SIDE_NONE && !(L.sr.kind == SIDE_CLOSEST_LIGHT && !trace_light_brdf);
                if (need)
                {
                    L.ro = L.sr.o; L.rd = L.sr.d; L.tmax = L.sr.tmax;
                    L.mode = L.sr.kind == SIDE_SHADOW ? TRACE_SHADOW : (L.sr.kind == SIDE_CLOSEST_LIGHT ? TRACE_CLOSEST : TRACE_ANY);
                    break;
                }
                L.stage++;
                continue;
            }
            // all four side rays resolved: continuation sample and path bookkeeping (:121-141)
            float bpdf;
            v3 ndir = V(0.0f, 0.0f, 0.0f);
            const col brdf = ct_sample(L.sf.m, L.sf.view, L.sf.n, ndir, bpdf, L.rng);
            if (L.bounce == 0) L.sample_color = L.sample_color + CO(L.sf.m.er, L.sf.m.eg, L.sf.m.eb);
            L.sample_color = L.sample_color + ((L.c0 + L.c1) + (L.c3 + L.c2)) * L.throughput;   // light = c0+c1 (:712), env = c3+c2 (:630)
            if (is_black(brdf) || bpdf < 1.0e-8f || isinf(bpdf)) { sample_done = true; break; }
            L.throughput = L.throughput * ((brdf * smax(0.0f, dot(ndir, L.sf.n))) / bpdf);
            L.bounce++;
            if (L.bounce >= P.max_bounces) { sample_done = true; break; }
            L.ro = L.sf.p + 1.0e-4f * L.sf.n; L.rd = ndir;
            L.mode = TRACE_CLOSEST; L.stage = 4;
            break;
        }

        // (5) sample / pixel bookkeeping
        if (sample_done)
        {
            L.final_color = L.final_color + L.sample_color;
            L.sample++;
            if (L.sample < P.spp) start_sample(P, L);
            else
            {
                const float n = (float)P.spp;
                const col mean = CO(L.final_color.r / n, L.final_color.g / n, L.final_color.b / n);   // operator/= divides (color.h:67-74)
                out_tiles[L.slot] = pixel_output(P.flags, fb_in_rowmajor, (size_t)L.y * P.cam.w + L.x, mean);
                have_pixel = false;
            }
        }
    }
    for (int off = 16; off > 0; off >>= 1) rays += __shfl_down_sync(FULL, rays, off);
    if (lane == 0 && rays) atomicAdd(ray_counter, rays);
}

// ---- K1: primary closest hit (parity hook + C2 traversal microbenchmark) -----------------------------------------------
template <int TL>
__global__ void __launch_bounds__(256) k_primary(SceneDev S, RenderParams P, int sample, int* __restrict__ prim_out, float* __restrict__ t_out)
{
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (warp >= P.n_rank_tiles * 8) return;
    const PixelSlot ps = unit_pixel(P, warp, lane);
    if (!ps.inside) return;
    float fx = (float)ps.x, fy = (float)ps.y;
    if (sample >= 0)
    {
        uint32_t rng = pixel_rng(ps.x, ps.y, P.spp);
        fx = ((float)ps.x + 0.5f) + xs_float(rng) - 1.0f;
        fy = ((float)ps.y + 0.5f) + xs_float(rng) - 1.0f;
    }
    v3 o, d;
    camera_ray(P.cam, fx, fy, o, d);
    Hit h;
    const bool found = trace_ray<TL>(S, o, d, 0.0f, TRACE_CLOSEST, h);
    const size_t idx = (size_t)ps.y * P.cam.w + ps.x;
    prim_out[idx] = found ? h.prim : -1;
    t_out[idx] = found ? h.t : -1.0f;
}

// ---- feature buffers for a denoiser (OIDN's "albedo" / "normal"): k x k stratified camera rays per pixel ------------------------
// The grid covers [x - 0.5, x + 0.5) like the beauty's jitter (x + 0.5 + r - 1, :88-89), so the guides are anti-aliased like the
// beauty; k = 1 is exactly k_primary's un-jittered ray. Per ray: the diffuse colour of the closest hit's material (the BRDF's base
// colour) and its geometric normal (hit_geometry: never flipped); a miss adds 0. Outputs are the means over the k^2 rays, the
// normal not renormalised (a partly covered pixel has length < 1). No RNG: deterministic.
template <int TL>
__global__ void __launch_bounds__(256) k_aov(SceneDev S, RenderParams P, int k, float* __restrict__ albedo_out, float* __restrict__ normal_out)
{
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (warp >= P.n_rank_tiles * 8) return;
    const PixelSlot ps = unit_pixel(P, warp, lane);
    if (!ps.inside) return;
    col a = CO(0.0f, 0.0f, 0.0f);
    v3 n = V(0.0f, 0.0f, 0.0f);
    for (int j = 0; j < k; j++)
        for (int i = 0; i < k; i++)
        {
            const float fx = (float)ps.x + (((float)i + 0.5f) / (float)k - 0.5f);
            const float fy = (float)ps.y + (((float)j + 0.5f) / (float)k - 0.5f);
            v3 o, d;
            camera_ray(P.cam, fx, fy, o, d);
            Hit h;
            if (!trace_ray<TL>(S, o, d, 0.0f, TRACE_CLOSEST, h)) continue;
            const MaterialDev m = S.mats[__ldg(S.mat_idx + h.prim)];
            a = a + CO(m.dr, m.dg, m.db);
            v3 p, hn;
            hit_geometry(S, h, o, d, p, hn);
            n = n + hn;
        }
    const float rays = (float)(k * k);
    const size_t idx = 3 * ((size_t)ps.y * P.cam.w + ps.x);
    if (albedo_out) { albedo_out[idx] = a.r / rays; albedo_out[idx + 1] = a.g / rays; albedo_out[idx + 2] = a.b / rays; }
    if (normal_out) { normal_out[idx] = n.x / rays; normal_out[idx + 1] = n.y / rays; normal_out[idx + 2] = n.z / rays; }
}

// ---- ray batches (BVH::intersect / FlattenedBVH::intersect replacement for tests and tools) ------------------------------
template <int TL>
__global__ void __launch_bounds__(256) k_trace_rays(SceneDev S, const float* __restrict__ rays6, int n, int any_hit,
                                                    int* __restrict__ prim_out, float* __restrict__ t_out, float* __restrict__ extra8)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float* r = rays6 + 6 * (size_t)i;
    const v3 o = V(r[0], r[1], r[2]), d = V(r[3], r[4], r[5]);
    Hit h;
    const bool found = trace_ray<TL>(S, o, d, 0.0f, any_hit ? TRACE_ANY : TRACE_CLOSEST, h);
    if (any_hit) { prim_out[i] = found ? 1 : 0; t_out[i] = found ? h.t : -1.0f; return; }
    prim_out[i] = found ? h.prim : -1;
    t_out[i] = found ? h.t : -1.0f;
    if (extra8)
    {
        float* e = extra8 + 8 * (size_t)i;
        if (found)
        {
            v3 p, nn;
            hit_geometry(S, h, o, d, p, nn);
            e[0] = p.x; e[1] = p.y; e[2] = p.z; e[3] = nn.x; e[4] = nn.y; e[5] = nn.z; e[6] = h.u; e[7] = h.v;
        }
        else { for (int k = 0; k < 8; k++) e[k] = 0.0f; }
    }
}

// ---- K4: tile-major (per-rank compact buffers, rank-major) -> row-major bottom-up RGBA --------------------------------------
__global__ void __launch_bounds__(256) k_untile(const float4* __restrict__ tiles, int tiles_per_rank_padded, int world, int only_rank,
                                                int w, int h, int tiles_x, int skew, float4* __restrict__ image)
{
    const int x = blockIdx.x * 16 + (threadIdx.x & 15);
    const int y = blockIdx.y * 16 + (threadIdx.x >> 4);
    if (x >= w || y >= h) return;
    const int tile_id = tile_number(x / kTileDim, y / kTileDim, tiles_x, skew);
    const int rank = tile_id % world, k = tile_id / world;
    if (only_rank >= 0 && rank != only_rank) return;
    const int lx = x % kTileDim, ly = y % kTileDim;
    const int sub = (ly / kPatchH) * 2 + (lx / kPatchW);
    const int lane = (ly % kPatchH) * kPatchW + (lx % kPatchW);
    const size_t src = ((size_t)(only_rank >= 0 ? 0 : rank) * tiles_per_rank_padded + k) * kTilePixels + sub * 32 + lane;
    image[(size_t)y * w + x] = tiles[src];
}

// K4 for B200RT_FLAG_LINEAR_TILES buffers: image (the incoming framebuffer) += mean radiance, tone map in place (:169-180)
__global__ void __launch_bounds__(256) k_untile_accumulate(const float4* __restrict__ tiles, int tiles_per_rank_padded, int world, int w, int h,
                                                           int tiles_x, int skew, float4* __restrict__ image)
{
    const int x = blockIdx.x * 16 + (threadIdx.x & 15);
    const int y = blockIdx.y * 16 + (threadIdx.x >> 4);
    if (x >= w || y >= h) return;
    const int tile_id = tile_number(x / kTileDim, y / kTileDim, tiles_x, skew);
    const int rank = tile_id % world, k = tile_id / world;
    const int lx = x % kTileDim, ly = y % kTileDim;
    const int sub = (ly / kPatchH) * 2 + (lx / kPatchW);
    const int lane = (ly % kPatchH) * kPatchW + (lx % kPatchW);
    const float4 m = tiles[((size_t)rank * tiles_per_rank_padded + k) * kTilePixels + sub * 32 + lane];
    const size_t i = (size_t)y * w + x;
    image[i] = tonemap(image[i], CO(m.x, m.y, m.z));
}

cudaError_t launch_untile_accumulate(const float4* tiles, int tiles_per_rank_padded, int world, int w, int h, float4* image, cudaStream_t stream)
{
    const int tiles_x = (w + kTileDim - 1) / kTileDim, tiles_y = (h + kTileDim - 1) / kTileDim;
    dim3 grid(tiles_x, tiles_y);
    k_untile_accumulate<<<grid, 256, 0, stream>>>(tiles, tiles_per_rank_padded, world, w, h, tiles_x, tile_skew(), image);
    return cudaGetLastError();
}

// fills a float array with one value (b200rt_trace_primary: "miss" for the pixels of other ranks)
__global__ void k_fill_f32(float* p, size_t n, float v)
{
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) p[i] = v;
}
cudaError_t launch_fill_f32(float* p, size_t n, float v, cudaStream_t stream)
{
    if (!n) return cudaSuccess;
    k_fill_f32<<<(unsigned int)std::min<size_t>((n + 255) / 256, 148 * 8), 256, 0, stream>>>(p, n, v);
    return cudaGetLastError();
}

__global__ void k_fill_f4(float4* p, size_t n, float4 v)
{
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) p[i] = v;
}
cudaError_t launch_fill_f4(float4* p, size_t n, float4 v, cudaStream_t stream)
{
    if (!n) return cudaSuccess;
    k_fill_f4<<<(unsigned int)std::min<size_t>((n + 255) / 256, 148 * 8), 256, 0, stream>>>(p, n, v);
    return cudaGetLastError();
}

// ---- output stage: the quantisation loop of write_image_png (source/image_io.cpp:165-182), 16 B in -> 4 B out per pixel -----
// Color pixel = image(i) * 255; tmp = clamp(pixel, 0, 255) -> unsigned char (truncation); flipY puts image row 0 (bottom) last.
__device__ __forceinline__ unsigned int quantise_channel(float v)
{
    const float p = v * 255.0f;
    const float c = p < 0.0f ? 0.0f : (p > 255.0f ? 255.0f : p);       // clamp() of image_io.cpp:157-162 (a NaN falls through)
    return (unsigned int)__float2int_rz(c) & 0xffu;
}
__global__ void __launch_bounds__(256) k_quantise_rgba8(const float4* __restrict__ image, int w, int h, int flip_y, uchar4* __restrict__ out)
{
    const int x = blockIdx.x * 32 + (threadIdx.x & 31);
    const int y = blockIdx.y * 8 + (threadIdx.x >> 5);
    if (x >= w || y >= h) return;
    const float4 p = image[(size_t)y * w + x];
    const int oy = flip_y ? h - 1 - y : y;
    out[(size_t)oy * w + x] = make_uchar4((unsigned char)quantise_channel(p.x), (unsigned char)quantise_channel(p.y),
                                          (unsigned char)quantise_channel(p.z), (unsigned char)quantise_channel(p.w));
}

// ---- parity hook: the RNG stream of one pixel (xorshift.h:10-31 seeded and warmed up as render_kernel.cpp:77-82) -----------------
__global__ void k_rng_stream(int x, int y, int spp, int n, uint32_t* state_out, float* floats_out)
{
    if (blockIdx.x || threadIdx.x) return;
    uint32_t s = pixel_rng(x, y, spp);
    *state_out = s;
    for (int i = 0; i < n; i++) floats_out[i] = xs_float(s);
}

cudaError_t launch_rng_stream(int x, int y, int spp, int n, uint32_t* state_out, float* floats_out, cudaStream_t stream)
{
    k_rng_stream<<<1, 32, 0, stream>>>(x, y, spp, n, state_out, floats_out);
    return cudaGetLastError();
}

// ---- parity hook: env_map_cdf_search (render_kernel.cpp:532-567) for a batch of values, with or without the guide table ----------
__global__ void __launch_bounds__(256) k_env_cdf_search(SceneDev S, const float* __restrict__ values, int n, int* __restrict__ xy)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int x, y;
    env_cdf_search(S, values[i], x, y);
    xy[2 * i] = x; xy[2 * i + 1] = y;
}

cudaError_t launch_env_cdf_search(const SceneDev& S, const float* values, int n, int* xy, cudaStream_t stream)
{
    if (n <= 0) return cudaSuccess;
    k_env_cdf_search<<<(n + 255) / 256, 256, 0, stream>>>(S, values, n, xy);
    return cudaGetLastError();
}

// ---- launchers ----------------------------------------------------------------------------------------------------------------
// SM count of the calling thread's current device (cached per device: one process may drive several GPU models)
int tile_skew()
{
    static const int v = []() { const char* e = getenv("B200RT_TILE_SKEW"); const int k = e ? atoi(e) : 0; return k < 0 ? 0 : k; }();
    return v;
}

int current_sm_count()
{
    static int cache[64] = {};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
    if (!cache[dev])
    {
        int n = 0;
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
        cache[dev] = n > 0 ? n : 148;
    }
    return cache[dev];
}
static int sm_count() { return current_sm_count(); }

cudaError_t launch_megakernel(const SceneDev& S, const RenderParams& P, const float4* fb_in_rowmajor, float4* out_tiles,
                              unsigned int* work_counter, unsigned long long* ray_counter, cudaStream_t stream)
{
    cudaError_t e = cudaMemsetAsync(work_counter, 0, sizeof(unsigned int), stream);
    if (e != cudaSuccess) return e;
    const int tl = traversal_layout(S, P.flags);
    int per_sm = 0;
    if (tl == TL_WIDE) cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_pathtrace_mega<TL_WIDE>, 256, 0);
    else if (tl == TL_DIAG) cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_pathtrace_mega<TL_DIAG>, 256, 0);
    else cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_pathtrace_mega<TL_AXIS>, 256, 0);
    if (per_sm <= 0) per_sm = 1;
    int grid = sm_count() * per_sm;                        // persistent: a whole number of resident CTAs per SM
    const int needed = P.rw > 0 ? (P.rw * P.rh + 255) / 256 : P.n_rank_tiles;      // one CTA's worth of lanes per 16x16 tile at most
    if (grid > needed) grid = needed;
    if (grid <= 0) return cudaSuccess;
    if (tl == TL_WIDE) k_pathtrace_mega<TL_WIDE><<<grid, 256, 0, stream>>>(S, P, fb_in_rowmajor, out_tiles, work_counter, ray_counter);
    else if (tl == TL_DIAG) k_pathtrace_mega<TL_DIAG><<<grid, 256, 0, stream>>>(S, P, fb_in_rowmajor, out_tiles, work_counter, ray_counter);
    else k_pathtrace_mega<TL_AXIS><<<grid, 256, 0, stream>>>(S, P, fb_in_rowmajor, out_tiles, work_counter, ray_counter);
    return cudaGetLastError();
}

cudaError_t launch_primary(const SceneDev& S, const RenderParams& P, int sample, int* prim_out, float* t_out, cudaStream_t stream)
{
    const int n_warps = P.n_rank_tiles * 8;
    if (n_warps <= 0) return cudaSuccess;
    const int grid = (n_warps * 32 + 255) / 256;
    const int tl = traversal_layout(S, P.flags, true);
    if (tl == TL_WIDE) k_primary<TL_WIDE><<<grid, 256, 0, stream>>>(S, P, sample, prim_out, t_out);
    else if (tl == TL_DIAG) k_primary<TL_DIAG><<<grid, 256, 0, stream>>>(S, P, sample, prim_out, t_out);
    else k_primary<TL_AXIS><<<grid, 256, 0, stream>>>(S, P, sample, prim_out, t_out);
    return cudaGetLastError();
}

cudaError_t launch_aov(const SceneDev& S, const RenderParams& P, int k, float* albedo_out, float* normal_out, cudaStream_t stream)
{
    const int n_warps = P.n_rank_tiles * 8;
    if (n_warps <= 0) return cudaSuccess;
    const int grid = (n_warps * 32 + 255) / 256;
    const int tl = traversal_layout(S, P.flags, true);
    if (tl == TL_WIDE) k_aov<TL_WIDE><<<grid, 256, 0, stream>>>(S, P, k, albedo_out, normal_out);
    else if (tl == TL_DIAG) k_aov<TL_DIAG><<<grid, 256, 0, stream>>>(S, P, k, albedo_out, normal_out);
    else k_aov<TL_AXIS><<<grid, 256, 0, stream>>>(S, P, k, albedo_out, normal_out);
    return cudaGetLastError();
}

cudaError_t launch_trace_rays(const SceneDev& S, const float* rays6, int n, int any_hit, int flags, int* prim_out, float* t_out,
                              float* extra8, cudaStream_t stream)
{
    if (n <= 0) return cudaSuccess;
    const int grid = (n + 255) / 256;
    const int tl = traversal_layout(S, flags);
    if (tl == TL_WIDE) k_trace_rays<TL_WIDE><<<grid, 256, 0, stream>>>(S, rays6, n, any_hit, prim_out, t_out, extra8);
    else if (tl == TL_DIAG) k_trace_rays<TL_DIAG><<<grid, 256, 0, stream>>>(S, rays6, n, any_hit, prim_out, t_out, extra8);
    else k_trace_rays<TL_AXIS><<<grid, 256, 0, stream>>>(S, rays6, n, any_hit, prim_out, t_out, extra8);
    return cudaGetLastError();
}

cudaError_t launch_quantise_rgba8(const float4* image, int w, int h, int flip_y, void* out_rgba8, cudaStream_t stream)
{
    if (w <= 0 || h <= 0) return cudaSuccess;
    dim3 grid((w + 31) / 32, (h + 7) / 8);
    k_quantise_rgba8<<<grid, 256, 0, stream>>>(image, w, h, flip_y, (uchar4*)out_rgba8);
    return cudaGetLastError();
}

cudaError_t launch_untile(const float4* tiles, int tiles_per_rank_padded, int world, int only_rank, int w, int h, float4* image,
                          cudaStream_t stream)
{
    const int tiles_x = (w + kTileDim - 1) / kTileDim, tiles_y = (h + kTileDim - 1) / kTileDim;
    dim3 grid(tiles_x, tiles_y);
    k_untile<<<grid, 256, 0, stream>>>(tiles, tiles_per_rank_padded, world, only_rank, w, h, tiles_x, tile_skew(), image);
    return cudaGetLastError();
}

} // namespace b200rt
