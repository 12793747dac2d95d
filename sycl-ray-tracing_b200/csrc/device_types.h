// POD structs shared by the host shim and the kernels.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace b200rt {

constexpr int kTileDim = 16;                 // image tiles are 16x16 pixels = 8 warp patches of 8x4
constexpr int kTilePixels = kTileDim * kTileDim;
constexpr int kPatchW = 8, kPatchH = 4;      // one warp = one 8x4 pixel patch
constexpr int kStackSize = 64;

// Which tile a rank's k-th tile is. Tiles are numbered L = 0 .. tiles_x * tiles_y - 1 and rank r owns the tiles with
// L % world == r; L = ty * tiles_x + (tx + skew * ty) % tiles_x walks every tile row from a start column that moves `skew`
// tiles per row (B200RT_TILE_SKEW, read once per process; RenderParams::tile_skew; the same map in distributed.py).
// 0, the default, is plain row-major numbering: a world that divides tiles_x (1920 / 16 = 120 tiles, 8 ranks) then owns
// whole tile COLUMNS. Measured on C3 / 8 GPUs (tools/rank_timing.py, every rank emulated on one GPU): columns give the ranks
// 125.6 ... 127.6 M rays and 94 ... 113 ms (mean 103); a skew of 5 (every 8 x 8 block of tiles holds every rank 8 times)
// evens the rays out to 126.0 ... 126.9 M and makes the ranks SLOWER, 104 ... 115 ms (mean 109): a rank's time is its chain
// of dependent passes (DESIGN.md 4.3), not its ray count, and a rank that sees vertical slabs of the scene keeps a smaller
// part of the BVH hot.
#ifdef __CUDACC__
#define B200RT_HD __host__ __device__
#else
#define B200RT_HD
#endif
B200RT_HD inline void tile_xy(int L, int tiles_x, int skew, int& tx, int& ty)
{
    ty = L / tiles_x;
    const int c = L - ty * tiles_x;
    tx = skew ? (c + tiles_x - (skew % tiles_x) * (ty % tiles_x) % tiles_x) % tiles_x : c;      // (tiles_x <= 2^15: the product fits)
}
B200RT_HD inline int tile_number(int tx, int ty, int tiles_x, int skew) { return ty * tiles_x + (skew ? (tx + (skew % tiles_x) * (ty % tiles_x) % tiles_x) % tiles_x : tx); }

struct MaterialDev   // SimpleMaterial (simple_material.h:6-13) without the junk alphas, two float4
{
    float er, eg, eb, metalness;
    float dr, dg, db, roughness;
};

struct SphereDev     // == Sphere (sphere.h:55-58)
{
    float cx, cy, cz, radius;
    int prim;
};

struct SceneDev
{
    const float4* axis;        // 4 float4 per inner node (AxisNode)
    const float4* diag;        // 4 float4 per inner node (DiagNode)
    const float4* wide;        // 5 float4 per node of the 8-ary quantised BVH (WideNode); null when the BVH has none
    const unsigned char* oct_lut; // [8][256]: hit mask by slot -> hit mask in front-to-back order for ray octant class o (bit s -> bit s ^ o)
    const float4* tris;        // 3 float4 per triangle, leaf order (LeafTriangle)
    const int* slot_of_prim;   // original triangle index -> slot in `tris`
    const int* mat_idx;        // per primitive (triangles, then spheres)
    const MaterialDev* mats;
    const int* emissive;       // original indices of emissive triangles
    const SphereDev* spheres;
    const float4* env;         // env_w * env_h RGBA
    const float* cdf;          // running luminance sum, row-major
    const float2* env_alias;   // per texel {acceptance probability, as_float(alias texel)}; null until b200rt_scene_build_env_alias
    const float* row_cdf;      // cdf[y * env_w + env_w - 1] for every row (the row search's probes, contiguous)
    const unsigned int* cdf_guide; // [cdf_guide_n + 2] lower bounds of the CDF search per value bucket (env_tables.cu); null = plain binary searches
    float cdf_guide_scale;     // bucket = min(cdf_guide_n - 1, (unsigned)(value * cdf_guide_scale))
    int cdf_guide_n;
    int n_tri, n_mats, n_emissive, n_spheres;
    int env_w, env_h;
    float cdf_total;
    int has_diag;
    int has_wide;
    int use_alias;             // this launch samples the env map through env_alias (B200RT_FLAG_ENV_ALIAS)
    unsigned int qmagic;       // 0x43000000 (see B200RT_Q in pt_device.cuh)
    int any_emissive_material; // some material has emission > 0 (else the BRDF->light MIS ray cannot contribute)
};

struct CameraDev   // Camera (camera.h:34-39) + frame size, as get_camera_ray uses them (render_kernel.cpp:56-73)
{
    float m[16];
    float fov_dist;
    int w, h;
};

struct RenderParams
{
    CameraDev cam;
    int spp, max_bounces;
    int rank, world;           // interleaved 16x16 tiles: tile number % world == rank (tile_xy / tile_number above)
    int tiles_x, tiles_y;
    int tile_skew;             // see tile_xy above
    int n_rank_tiles;          // tiles owned by this rank
    int flags;
    // region mode (b200rt_render_region, megakernel only): slots are the pixels of the rectangle [rx0, rx0 + rw) x [ry0, ry0 + rh)
    // of the frame in row-major order instead of this rank's tiles; rw == 0 = off
    int rx0, ry0, rw, rh;
    // progressive accumulation (b200rt_accum_*, wavefront / persistent integrators): this launch renders samples
    // [sample_begin, sample_end) of every pixel. spp stays the TOTAL sample count of the frame: it seeds the per-pixel RNG
    // (31 + x*y*spp, render_kernel.cpp:77). acc_rng / acc_sum (indexed like the tile buffer) carry each pixel's generator state
    // and radiance sum from one launch to the next; null = an ordinary one-shot frame (sample_begin = 0, sample_end = spp).
    int sample_begin, sample_end;
    uint32_t* acc_rng;
    float4* acc_sum;
};

// wavefront integrator state: one slot per pixel of this rank's tile-major buffer (SoA, HBM resident)
struct WfBuffers
{
    int n_slots;
    int tile_stride, tile_offset;             // slot s of this group writes out_tiles[((s >> 8) * tile_stride + tile_offset) * 256 + (s & 255)]
    uint32_t* rng; int* sample; int* bounce; int* flags;
    float4* final_c; float4* sample_c; float4* thr; float4* thr_next;
    float4* ray_o; float4* ray_d;             // [5 * n_slots]: k * n_slots + slot; k = 0..3 side rays, 4 = path ray; .w = tmax / ray kind
    float4* side_w;                           // [4 * n_slots]: MIS-weighted contribution if unoccluded (.w = direction pdf for k = 1)
    float4* res;                              // [5 * n_slots]: {t, primitive (closest hit) | occlusion flag, triangle slot, -} of each ray
    unsigned int* queue;                      // [5 * n_slots]: (slot << 3) | k
    unsigned int* counters;                   // [2] = pixels still rendering, [3], [4] = ping-pong queue lengths
    unsigned long long* rays_total;
};

constexpr int kMaxWfGroups = 8;

// one interleaved tile group of the wavefront integrator: its state, stream and polling resources
struct WfGroup
{
    WfBuffers buf;
    cudaStream_t stream;
    cudaEvent_t poll_event, join_event;
    unsigned int* host_active;      // pinned
};

} // namespace b200rt
