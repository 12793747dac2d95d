/* b200rt.h — the drop-in boundary: a C ABI (plain pointers and sizes, no torch / C++ types) over the B200-native
 * implementation of the reference's per-pixel path-tracing hot path.
 *
 * Every entry point cites the reference interface it replaces (file:line in TomClabault/SYCL-ray-tracing).
 * The reference has no FFI of its own (it is one C++ process, source/main.cpp:63-128); the binding a maintainer adds
 * is the C++ `RenderKernel` in sycl-ray-tracing_b200/host/dropin/ (see INTEGRATION.md), or ctypes
 * (sycl-ray-tracing_b200/binding.py).
 *
 * All functions return 0 on success and a non-zero code on failure; b200rt_last_error() describes the last failure
 * of the calling thread. There is NO CPU fallback: without a CUDA device every compute entry point fails with
 * B200RT_ERR_CUDA.
 *
 * Layout contracts (trivially-copyable reference structs can be passed straight through with vector::data()):
 *   triangles   : 9 floats  {a.xyz, b.xyz, c.xyz}                         == Triangle        include/triangle.h:67
 *   materials   : 10 floats {emission rgba, diffuse rgba, metal, rough}   == SimpleMaterial  include/simple_material.h:6-13
 *   spheres     : 20 bytes  {center xyz, radius, int primitive_index}     == Sphere          include/sphere.h:55-58
 *   camera      : 17 floats {view_matrix row-major 4x4, fov_dist}         <- Camera          include/camera.h:34-39
 *   framebuffer : w*h*4 floats RGBA, row-major, row 0 = BOTTOM row        == Image           include/image.h:25-178
 *   env map     : env_w*env_h*4 floats RGBA, row-major                    == Image (skysphere), CDF: utils.cpp:126-142
 */
#ifndef B200RT_H
#define B200RT_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200RT_OK 0
#define B200RT_ERR_ARG 1
#define B200RT_ERR_CUDA 2
#define B200RT_ERR_ALLOC 3

typedef struct b200rt_bvh b200rt_bvh;      /* host-side flattened BVH (the re-laid-out FlattenedBVH) */
typedef struct b200rt_scene b200rt_scene;  /* device-resident scene: triangles, BVH, materials, lights, env map */

/* ---- FlattenedBVH -------------------------------------------------------------------------------------------------
 * Replaces BVH::BVH + BVH::flatten() (source/bvh.cpp:19-60, include/bvh.h:211-250) and the 128-byte AoS
 * FlattenedBVH::FlattenedNode (include/flattened_bvh.h:25-39). New layout, two parallel 64-byte-aligned streams with
 * one record per INNER node, each record describing BOTH children (so one 64 B fetch tests two volumes):
 *   axis[i]  : 16 floats {L.lo.xyz, L.hi.xyz, R.lo.xyz, R.hi.xyz, int L.ref, int R.ref, int L.count, int R.count}
 *              = the 3 axis-aligned slabs of the 7-plane volume (PLANE_NORMALS[0..2], source/bvh.cpp:8-16)
 *   diag[i]  : 16 floats {L.near[3..6], L.far[3..6], R.near[3..6], R.far[3..6]}
 *              = the 4 diagonal slabs (PLANE_NORMALS[3..6]); only fetched when an axis test passes
 *   ref >= 0 : index of an inner node; ref <  0 : leaf, ~ref = (first << 4) | count: triangles [first, first + count) of the leaf-ordered stream
 *   tris[j]  : 12 floats {a.xyz, as_float(original index), e1.xyz = b-a, 0, e2.xyz = c-a, 0}   (3 x float4)
 * Leaves hold (first, count) ranges, so the >8-triangle leaf overflow of the reference (bvh.h:226 vs
 * flattened_bvh.h:35) cannot happen.
 * On top of the same binary tree the builder emits the layout the kernels traverse by default: an 8-ary BVH of
 * 80-byte nodes whose 8 child boxes are quantised to one byte per plane (csrc/bvh_build.h WideNode,
 * csrc/pt_device.cuh); both layouts index the same leaf-ordered triangle stream. */
typedef struct b200rt_bvh_options
{
    int max_leaf_size;     /* SAH may stop at <= this many triangles per leaf; default 3, max 15 (the 8-ary BVH needs <= 3) */
    int sah_bins;          /* default 16 */
    int use_diag_slabs;    /* 1: emit the 4 diagonal slabs (7-plane volumes); 0: axis slabs only. default 1 */
    int num_threads;       /* builder threads; 0 = all */
} b200rt_bvh_options;

typedef struct b200rt_bvh_info
{
    int n_triangles, n_inner_nodes, n_leaves, max_leaf_size, max_depth, has_diag_slabs;
    double build_seconds;
    double sah_cost;
    int n_wide_nodes;      /* nodes of the 8-ary quantised BVH (0 when max_leaf_size > 3: its leaves hold at most 3 triangles) */
    int wide_max_depth;
} b200rt_bvh_info;

void b200rt_bvh_default_options(b200rt_bvh_options* opts);
int b200rt_bvh_build(const float* tri_xyz9, int n_tri, const b200rt_bvh_options* opts_or_null, b200rt_bvh** out);
/* Same product, built on the GPU (`device`; < 0 = current): Morton-order linear BVH (sort, parallel radix tree, bottom-up
 * fit), collapsed level by level into the 8-ary layout; no diagonal slabs (has_diag_slabs = 0). Tree quality is below
 * the host builder's binned SAH (slower traversal), construction is two orders of magnitude faster — for scenes where
 * BVH::BVH (source/bvh.cpp:19-60: sequential insert, ~13 s with the host SAH builder at 20 M triangles) dominates.
 * Host pointer in, host arrays out (like b200rt_bvh_build); no CPU fallback. */
int b200rt_bvh_build_device(const float* tri_xyz9, int n_tri, int device, b200rt_bvh** out);
int b200rt_bvh_get_info(const b200rt_bvh* bvh, b200rt_bvh_info* out);
/* borrowed pointers into the host arrays described above; valid until b200rt_bvh_destroy  (FlattenedBVH::get_nodes, flattened_bvh.h:43-44) */
int b200rt_bvh_get_arrays(const b200rt_bvh* bvh, const float** axis16, const float** diag16, const float** tris12);
/* the 8-ary layout: *nodes80 = n_nodes records of 80 bytes (layout: csrc/bvh_build.h WideNode, decoding: csrc/pt_device.cuh);
 * borrowed, valid until b200rt_bvh_destroy; n_nodes = 0 when the BVH has none (max_leaf_size > 3) */
int b200rt_bvh_get_wide_nodes(const b200rt_bvh* bvh, const void** nodes80, int* n_nodes);
/* structural self-check (every triangle in exactly one leaf, every child volume contains its triangles): 0 = sound */
int b200rt_bvh_check(const b200rt_bvh* bvh, const float* tri_xyz9, int n_tri);
void b200rt_bvh_destroy(b200rt_bvh* bvh);

/* ---- scene ---------------------------------------------------------------------------------------------------------
 * Replaces the 13-argument RenderKernel constructor's borrowed buffers (include/render_kernel.h:24-46,
 * source/main.cpp:95-106): everything is copied to HBM once and stays resident across renders.
 * tri_material has n_material_indices >= n_tri entries (analytic spheres index past the triangles, main.cpp:19-31).
 * env_cdf may be NULL: it is then computed on the device exactly as Utils::compute_env_map_cdf does (utils.cpp:126-142: the
 * same serial float additions, bit for bit).
 * bvh may be NULL: one is built with default options (host SAH builder; from 5 M triangles on, the device builder).
 * device < 0 = the calling thread's current CUDA device. The calling thread's current device is left unchanged by every call. */
int b200rt_scene_create(const float* tri_xyz9, int n_tri,
                        const int* tri_material, int n_material_indices,
                        const float* materials10, int n_materials,
                        const int* emissive_tri, int n_emissive,
                        const void* spheres20, int n_spheres,
                        const float* env_rgba, int env_w, int env_h, const float* env_cdf_or_null,
                        const b200rt_bvh* bvh_or_null, int device,
                        b200rt_scene** out);
/* Multi-GPU behind the boundary (SURVEY §8e): the same scene replicated on n_devices GPUs of this process (devices_or_null ==
 * NULL: devices 0 .. n_devices-1). b200rt_render / b200rt_render_rgba8 on such a scene cut the frame into interleaved 16x16
 * tiles (tile_id % n_devices), render every share on its own device from its own host thread, gather the per-rank tile
 * buffers on devices[0] with one peer copy per rank (NVLink) and do `framebuffer += final; tone map`
 * (render_kernel.cpp:169-180) there — the incoming framebuffer is honoured and the result equals the 1-GPU frame bit for bit.
 * The BVH is built once. A device may be listed more than once (several ranks then share it: how a one-GPU box exercises
 * this path). env_channels: 4 = RGBA (Image), 3 = the RGB triplets stbi_loadf returns, expanded to RGBA with
 * alpha 0 on the device (Utils::read_image_float, utils.cpp:113-121). */
int b200rt_scene_create_multi(const float* tri_xyz9, int n_tri,
                              const int* tri_material, int n_material_indices,
                              const float* materials10, int n_materials,
                              const int* emissive_tri, int n_emissive,
                              const void* spheres20, int n_spheres,
                              const float* env_pixels, int env_channels, int env_w, int env_h, const float* env_cdf_or_null,
                              const b200rt_bvh* bvh_or_null, const int* devices_or_null, int n_devices,
                              b200rt_scene** out);
int b200rt_scene_device_count(const b200rt_scene* scene);
void b200rt_scene_destroy(b200rt_scene* scene);
/* replace the materials in place (C4 roughness/metalness sweeps re-use the resident geometry) */
int b200rt_scene_set_materials(b200rt_scene* scene, const float* materials10, int n_materials);
/* Builds, ON THE DEVICE (csrc/env_tables.cu: three prefix sums and two binary searches per texel, in double), the alias table
 * of the environment map's luminance that B200RT_FLAG_ENV_ALIAS samples from (8 bytes per texel). Replaces
 * Utils::compute_env_map_cdf (utils.cpp:126-142) + env_map_cdf_search (render_kernel.cpp:532-567) for callers that opt in. */
int b200rt_scene_build_env_alias(b200rt_scene* scene);
/* the device-built table, downloaded: env_w*env_h acceptance probabilities and alias texels, *total_out = the luminance sum */
int b200rt_scene_get_env_alias(b200rt_scene* scene, float* prob_out, int* alias_out, double* total_out_or_null);
/* the running-sum CDF the integrator searches (the caller's, or — env_cdf_or_null == NULL at creation — the one the device
 * computed in the reference's serial float order, Utils::compute_env_map_cdf, utils.cpp:126-142): env_w*env_h floats */
int b200rt_scene_get_env_cdf(b200rt_scene* scene, float* cdf_out);
/* the same table on the host, for callers / tests that want to look at it: env_w*env_h acceptance probabilities and alias
 * texels; *total_out (may be NULL) = the exact luminance sum the probabilities are normalised with. Host-only, no GPU needed. */
int b200rt_env_alias_table(const float* env_rgba, int env_w, int env_h, float* prob_out, int* alias_out, double* total_out);
int b200rt_scene_get_bvh_info(const b200rt_scene* scene, b200rt_bvh_info* out);
size_t b200rt_scene_device_bytes(const b200rt_scene* scene);

/* ---- ingest ----------------------------------------------------------------------------------------------------------------------
 * b200rt_obj_load replaces Utils::parse_obj (source/utils.cpp:16-98: rapidobj parse + Triangulate -> ParsedOBJ): the same triangle
 * list in the same order (quads cut along their shorter diagonal like rapidobj; larger polygons fanned), material indices shifted
 * by one (slot 0 = the default material, emission (1, 0, 1)), roughness clamped to >= 1e-2, illum 0 -> roughness 1 / metalness 0,
 * emissive triangles listed. The arrays are exactly what b200rt_scene_create[_multi] takes; borrowed, valid until b200rt_obj_destroy.
 * b200rt_hdr_load replaces the stbi_loadf call of Utils::read_image_float (utils.cpp:100-124) for Radiance .hdr files: RGB triplets
 * (pass them to b200rt_scene_create_multi with env_channels = 3: the RGBA expansion happens on the device), row 0 = bottom row
 * when flip_y != 0, as the reference loads it. Host code. */
typedef struct b200rt_obj b200rt_obj;
int b200rt_obj_load(const char* path, b200rt_obj** out);
int b200rt_obj_get(const b200rt_obj* obj, const float** tri_xyz9, int* n_tri, const int** tri_material, const float** materials10,
                   int* n_materials, const int** emissive_tri, int* n_emissive);
void b200rt_obj_destroy(b200rt_obj* obj);
typedef struct b200rt_hdr b200rt_hdr;
int b200rt_hdr_load(const char* path, int flip_y, b200rt_hdr** out);
int b200rt_hdr_get(const b200rt_hdr* hdr, const float** rgb, int* width, int* height);
void b200rt_hdr_destroy(b200rt_hdr* hdr);

/* ---- rendering -------------------------------------------------------------------------------------------------------- */
#define B200RT_INTEGRATOR_MEGAKERNEL 0   /* persistent lanes, one pixel at a time per lane, single trace site */
#define B200RT_INTEGRATOR_WAVEFRONT 1    /* path-regeneration wavefront: shade / trace kernel pairs over tile groups (default) */
#define B200RT_INTEGRATOR_PERSISTENT 2   /* the wavefront without its frame-wide barrier: one launch per frame, every warp shades and traces
                                            its own K * 32 pixel slots and pulls new pixels as they finish (csrc/persist.cu) */

#define B200RT_FLAG_FB_IS_ZERO 1         /* caller guarantees the framebuffer is Color::Black(): skip its upload */
#define B200RT_FLAG_SKIP_DEAD_RAYS 2     /* skip rays whose result provably cannot change the image (see DESIGN.md) */
#define B200RT_FLAG_DIAG_SLABS 4         /* traverse with all 7 planes (test the 4 diagonal slabs after the 3 axis slabs); default: axis slabs
                                            only — measured faster on every workload, see DESIGN.md */
#define B200RT_FLAG_SIMPLE_TRACE 8       /* wavefront ablation: one-ray-per-lane grid-stride trace kernel instead of the default persistent
                                            kernel (per-lane ray refill + warp phase vote), see DESIGN.md */

#define B200RT_FLAG_BVH2 16              /* ablation: traverse the binary two-children-per-record layout instead of the default 8-ary
                                            quantised BVH (B200RT_FLAG_DIAG_SLABS implies it) */

#define B200RT_FLAG_BVH8 64              /* b200rt_trace_primary: use the 8-ary layout too (coherent camera rays default to the binary one, which is
                                            faster for them; every other entry point already defaults to the 8-ary layout) */
#define B200RT_FLAG_TIME_KERNELS 128     /* wavefront: bracket every trace and shade launch with CUDA events and report the sums in the stats
                                            struct; the tile groups then run one after the other: a measurement mode, slower than the default */
#define B200RT_FLAG_ENV_ALIAS 32         /* sample_environment_map's texel pick (render_kernel.cpp:532-567, two dependent binary searches over the float
                                            running-sum CDF, ~21 dependent loads) is replaced by one alias-table lookup with the same single RNG draw.
                                            Same per-texel probability lum/total in exact arithmetic, different draw -> texel map: the image agrees
                                            with the default statistically, not bit for bit. Needs b200rt_scene_build_env_alias(). */

#define B200RT_FLAG_TIME_INLINE 512      /* wavefront: as B200RT_FLAG_TIME_KERNELS, but nothing is serialised — every launch is bracketed by events on its own
                                            group stream while the tile groups overlap as in a normal frame, and the events are read after the frame.
                                            stats: trace_ms / shade_ms = summed launch durations (they overlap: the sum may exceed the frame),
                                            trace_union_ms = time during which at least one trace kernel was running */
#define B200RT_FLAG_WF_PASSES_ONLY 1024  /* wavefront ablation: trace / shade passes to the last pixel; the default hands the last few pixels of
                                            each tile group to one barrier-free tail launch (csrc/persist.cu wf_tail) instead */
/* flag bits 2048 and 4096 are retired: the library ignores them, and they must not be reused */
#define B200RT_FLAG_LINEAR_TILES 256     /* b200rt_render_tiles_device: the tile buffer receives each pixel's mean radiance (`final_color / spp`,
                                            render_kernel.cpp:167) instead of the tone-mapped value; b200rt_untile_accumulate_device then does
                                            `framebuffer += final; tone map` (:169-180) on the gathering device, so the incoming framebuffer is
                                            honoured on the multi-GPU path without shipping it to every rank */

typedef struct b200rt_render_options
{
    int integrator;       /* B200RT_INTEGRATOR_* */
    int flags;            /* B200RT_FLAG_* */
    int rank, world;      /* this process renders the 16x16 tiles with tile_id % world == rank (default 0, 1) */
} b200rt_render_options;

typedef struct b200rt_stats
{
    unsigned long long rays;        /* INTERSECT_SCENE-equivalent queries traced (render_kernel.cpp:504) */
    unsigned long long samples;     /* camera samples = pixels * spp rendered by this call */
    double kernel_ms;               /* CUDA-event time of the render kernels on the launching stream */
    double total_ms;                /* including host<->device copies done by this call */
    int gpu_launches;               /* kernels launched by this call */
    unsigned long long h2d_bytes, d2h_bytes;
    /* only with B200RT_FLAG_TIME_KERNELS (wavefront integrator): CUDA-event time of every trace / shade launch, summed */
    double trace_ms, shade_ms;
    int trace_launches, shade_launches;
    double trace_union_ms;          /* B200RT_FLAG_TIME_INLINE only */
    double tail_ms;                 /* B200RT_FLAG_TIME_INLINE only: summed duration of the barrier-free tail launches (csrc/persist.cu) */
    int tail_launches;
} b200rt_stats;

void b200rt_default_render_options(b200rt_render_options* opts);

/* Replaces RenderKernel::set_camera + RenderKernel::render (include/render_kernel.h:48,57;
 * source/render_kernel.cpp:189-211 -> ray_trace_pixel :75-181): framebuffer_rgba_inout[i] += mean radiance, then
 * tone-mapped in place (exposure 1.5, gamma 2.2, :167-180). Host pointers; blocking. */
int b200rt_render(b200rt_scene* scene, const float* camera17, int width, int height, int spp, int max_bounces,
                  float* framebuffer_rgba_inout, const b200rt_render_options* opts_or_null, b200rt_stats* stats_or_null);

/* Same as b200rt_render, but the frame leaves the GPU as RGBA8 — the bytes write_image_png would put into the PNG
 * (source/image_io.cpp:165-182: x255, clamp, truncate; flip_y != 0 writes the bottom row last): 4 B/pixel over PCIe instead of
 * 16. framebuffer_rgba_in_or_null is the incoming Image (NULL = Color::Black()); it is read, never written. */
int b200rt_render_rgba8(b200rt_scene* scene, const float* camera17, int width, int height, int spp, int max_bounces,
                        const float* framebuffer_rgba_in_or_null, int flip_y, unsigned char* out_rgba8,
                        const b200rt_render_options* opts_or_null, b200rt_stats* stats_or_null);

/* Replaces RenderKernel::ray_trace_pixel(x, y) (include/render_kernel.h:56, source/render_kernel.cpp:75-181) and the
 * DEBUG_PIXEL single-pixel mode (:186-197) for a rectangle of pixels [x0, x1) x [y0, y1) of the width x height frame: the
 * pixels keep the frame's coordinates, hence its camera rays and RNG seeds (31 + x*y*spp), so a crop equals the same
 * pixels of the full render bit for bit. out_rgba: (y1-y0)*(x1-x0)*4 floats, row-major, row 0 = y0; the value each pixel
 * would hold after render() on a Color::Black() framebuffer. One pixel: x1 = x0 + 1, y1 = y0 + 1. */
int b200rt_render_region(b200rt_scene* scene, const float* camera17, int width, int height, int spp, int max_bounces,
                         int x0, int y0, int x1, int y1, float* out_rgba, const b200rt_render_options* opts_or_null,
                         b200rt_stats* stats_or_null);

/* ---- progressive accumulation ----------------------------------------------------------------------------------------------------
 * The reference's render() adds the frame's mean radiance to the Image and tone-maps it IN PLACE (render_kernel.cpp:167-180), so a
 * second render() on the same Image is not an accumulation (SURVEY §5). An accumulator keeps every pixel's generator state and linear
 * radiance sum on the device instead, so the samples of a frame can be streamed in chunks and looked at in between:
 *   b200rt_accum_create   fixes scene, camera, frame size, the TOTAL spp (it seeds the per-pixel RNG: 31 + x*y*spp, :77) and max_bounces
 *   b200rt_accum_add      renders the next n_samples samples of every pixel, continuing each pixel's RNG stream where it stopped
 *   b200rt_accum_resolve  framebuffer_out = tone_map(framebuffer_in (NULL = Color::Black()) + sum / samples so far); any time, any number of times
 *   b200rt_accum_resolve_rgba8  the same frame as b200rt_accum_resolve, quantised on the device to the bytes write_image_png would write
 *                         (as b200rt_render_rgba8: image_io.cpp:165-182, flip_y != 0 writes the bottom row last): 4 B/pixel over PCIe
 *                         instead of 16, which is what a preview wants (33 MB instead of 133 MB per 4K resolve)
 * After spp_total samples — in any chunking — the resolved frame equals b200rt_render(spp_total) bit for bit, and the RGBA8 resolve
 * equals b200rt_render_rgba8(spp_total) byte for byte.
 * On a multi-device scene (b200rt_scene_create_multi) the state is split like a frame: rank d keeps the pixels of the interleaved 16x16
 * tiles it owns (tile_id % n_devices == d) on its own device, and a rank owns none when the frame has fewer tiles than there are
 * devices. An add runs every rank's share of the chunk at once, one host thread per device, with no traffic between devices; a
 * resolve gathers the ranks' tiles on the scene's first device (one peer copy per rank) and tone-maps there. Either way the
 * results are the single-device accumulator's, bit for bit. The state is the accumulator's own: b200rt_render on the same scene
 * between two adds does not disturb it.
 * opts: integrator WAVEFRONT or PERSISTENT, flags as b200rt_render; rank/world must stay 0/1. A refused add changes nothing. Host
 * pointers; blocking. Destroy an accumulator before its scene. */
typedef struct b200rt_accum b200rt_accum;
int b200rt_accum_create(b200rt_scene* scene, const float* camera17, int width, int height, int spp_total, int max_bounces, b200rt_accum** out);
int b200rt_accum_add(b200rt_accum* acc, int n_samples, const b200rt_render_options* opts_or_null, b200rt_stats* stats_or_null);
int b200rt_accum_samples(const b200rt_accum* acc);
int b200rt_accum_resolve(b200rt_accum* acc, const float* framebuffer_rgba_in_or_null, float* framebuffer_rgba_out);
int b200rt_accum_resolve_rgba8(b200rt_accum* acc, const float* framebuffer_rgba_in_or_null, int flip_y, unsigned char* out_rgba8);
void b200rt_accum_destroy(b200rt_accum* acc);

/* ---- geometry updates ------------------------------------------------------------------------------------------------------------
 * New vertex positions for the scene's triangles, in place: no rebuild, no new upload of materials, lights or environment tables,
 * and the wavefront state and every accumulator stay. tri_xyz9 holds n_tri triangles in the creation layout; triangle i replaces
 * triangle i given at creation.
 *   Fixed topology: n_tri must equal the scene's triangle count. Triangle order, material indices, the emissive list, spheres and the
 *     environment stay as they are. The tree keeps its shape (which triangles share a leaf, which subtrees share a node) and every
 *     box of both layouts, the diagonal slabs and the triangle stream are recomputed on the device from the new vertices, one tree
 *     level per launch, deepest first.
 *   Exact: closest hits do not depend on the tree's shape (ties go to the lowest original index), so after an update every entry point
 *     returns bit for bit what a scene freshly created from the new vertices returns: framebuffers, RGBA8, regions, feature buffers,
 *     primary maps, closest-hit ray batches, any-hit flags and ray counts (an any-hit t is whichever hit the traversal meets first,
 *     which depends on the tree's shape, for a fresh scene too). Only the speed differs: a tree refitted far from the shape it was
 *     built for has larger, more overlapping boxes. b200rt_scene_get_bvh_info then reports the refitted tree's sah_cost (sum over the binary records of child
 *     area / root area, leaves weighted by their triangle count, in double), so a caller can watch it grow and rebuild the tree
 *     (b200rt_scene_rebuild_bvh below).
 *   Refusals change nothing: B200RT_ERR_ARG for a NULL pointer, a wrong n_tri, or any NaN or +-Inf coordinate (no box can bound it;
 *     the check is the first device pass and runs before anything resident is written).
 *   Blocking, like b200rt_scene_set_materials. Multi-device scenes: every replica is updated on its own device, from one host thread
 *     each, and the replicas stay byte-identical.
 *   Accumulators survive an update, and samples added afterwards see the new geometry. An accumulation that spans an update mixes
 *     both geometries in one frame; that is the caller's choice.
 * stats (may be NULL): kernel_ms, total_ms, gpu_launches, h2d_bytes.
 * _device: dev_tri_xyz9 is device memory of the scene's first device; the update is ordered after the caller's prior work on
 * cuda_stream (a cudaStream_t of that device; NULL = legacy default stream), then synchronises. Vertices produced on the GPU never
 * cross PCIe; other replicas receive them device to device. The caller's current device is restored. */
int b200rt_scene_update_triangles(b200rt_scene* scene, const float* tri_xyz9, int n_tri, b200rt_stats* stats_or_null);
int b200rt_scene_update_triangles_device(b200rt_scene* scene, const void* dev_tri_xyz9, int n_tri,
                                         void* cuda_stream, b200rt_stats* stats_or_null);
/* Rebuilds the scene's BVH in place from new vertex positions, for geometry that has moved too far for a refit to serve it well (a
 * refitted tree keeps its shape, and its boxes grow and overlap as the motion departs from the shape it was built for; sah_cost
 * need not show it: a rigid rotation keeps it flat). Everything else stays resident: materials, the emissive list, spheres, the
 * environment and its tables, the alias table, the wavefront and persistent slot state, and every accumulator. tri_xyz9 holds n_tri
 * triangles in the creation layout; triangle i replaces triangle i, and n_tri must equal the scene's triangle count.
 *   The tree is replaced, not refitted: afterwards the scene holds exactly what b200rt_bvh_build_device returns for the new vertices,
 *     byte for byte (8-ary nodes, triangle stream, binary records, the bvh_info counts and depths), whichever builder serves it: the
 *     clustering build, the Morton radix tree for inputs clustering gives up on, or the host SAH builder for at most 3 triangles and
 *     for inputs both device builders decline. A device-built tree has no diagonal slabs, so a host-built scene that is rebuilt
 *     reports has_diag_slabs = 0, and B200RT_FLAG_DIAG_SLABS then traverses the axis slabs, as on any device-built scene.
 *   Exact, as an update: every entry point then returns bit for bit what a scene freshly created from the new vertices returns (an
 *     any-hit t excepted). b200rt_scene_get_bvh_info reports the new tree; build_seconds is the rebuild's wall time and sah_cost the
 *     refit's device reduction over the new binary records, so it compares with a refitted tree's.
 *   On the device: the build reads the vertices on the scene's first device and writes the new arrays there. Only the builder's
 *     top-level sweep (at most ~1 000 clusters) and the few outsized triangles of the top level (at most 45) cross PCIe, and the
 *     extent pass's and the SAH's results; no tree-sized array does (the host builder's inputs excepted, which are small).
 *   Refusals change nothing: B200RT_ERR_ARG for a NULL pointer, a wrong n_tri, a NaN or +-Inf coordinate (found by the extent pass
 *     before anything is built) or more than 2^27 - 1 triangles. The new arrays are built beside the old ones and swapped in only
 *     when every replica has its copy, so after a refusal, a failed allocation or a CUDA error the scene keeps its old tree, byte for
 *     byte. Peak device memory holds both trees.
 *   Blocking. Multi-device scenes: the tree is built once on the first device and copied device to device to every replica, which
 *     stay byte-identical. The old arrays are freed with cudaFree, which waits for work already queued on the device: a render that
 *     an earlier stream is still running when the rebuild returns finishes on the old tree.
 *   Accumulators survive, as for an update. A refit (b200rt_scene_update_triangles) afterwards refits the new tree.
 * stats (may be NULL): kernel_ms (CUDA events around the extent pass, the build and the SAH on the build's stream; it includes the
 * builder's host round trips: the top-level sweep and its level-by-level size reads), total_ms, gpu_launches (a library sort or scan
 * counts as one), h2d_bytes and d2h_bytes (the vertices when they come from the host, and every small copy of the build).
 * _device: dev_tri_xyz9 is device memory of the scene's first device, read in place; the rebuild is ordered after the caller's prior
 * work on cuda_stream (a cudaStream_t of that device; NULL = legacy default stream) and runs on it. The caller's current device is
 * restored. */
int b200rt_scene_rebuild_bvh(b200rt_scene* scene, const float* tri_xyz9, int n_tri, b200rt_stats* stats_or_null);
int b200rt_scene_rebuild_bvh_device(b200rt_scene* scene, const void* dev_tri_xyz9, int n_tri,
                                    void* cuda_stream, b200rt_stats* stats_or_null);
/* Test / inspection hook: downloads replica `replica`'s resident arrays. Sizes from b200rt_scene_get_bvh_info: n_wide_nodes records
 * of 80 bytes (csrc/bvh_build.h WideNode), n_inner_nodes binary records of 16 floats each for axis and diag (diag is written only
 * when has_diag_slabs), n_triangles leaf records of 12 floats. Any output may be NULL. */
int b200rt_scene_get_bvh_arrays(b200rt_scene* scene, int replica, void* wide80_out, float* axis16_out,
                                float* diag16_out, float* tris12_out);

/* Parity hook for xorshift32_generator (include/xorshift.h:10-31) as ray_trace_pixel seeds it (render_kernel.cpp:77-82):
 * *state_out = the generator state of pixel (x, y) after the 10 warm-up draws (seed 31 + x*y*spp in wrapping int arithmetic),
 * floats_out[0..n) = the next n floats. Runs on the calling thread's current device. */
int b200rt_rng_stream(int x, int y, int spp, int n, uint32_t* state_out, float* floats_out);

/* Parity hook for env_map_cdf_search (render_kernel.cpp:532-567): the texel (x, y) the reference's two binary searches pick for each of
 * n values (value = draw * cdf total), as the integrators evaluate it. use_guide != 0: through the guide table built at scene creation
 * (the default path when the CDF is non-decreasing); 0: the reference's plain searches. Both must agree. xy_out: 2*n ints. Host pointers. */
int b200rt_env_cdf_search(b200rt_scene* scene, const float* values, int n, int use_guide, int* xy_out);

/* Page-locked host memory for framebuffers / result arrays: copies from and to such buffers run at the full PCIe rate and are
 * not staged. Pageable buffers are accepted everywhere too (staged through the library's own pinned chunks). */
int b200rt_host_alloc(size_t bytes, void** out);
void b200rt_host_free(void* p);

/* Parity hook = RenderKernel::get_camera_ray + INTERSECT_SCENE for every pixel (render_kernel.cpp:56-73, :504-511).
 * sample < 0: un-jittered rays through (float)x,(float)y; sample >= 0: the jittered ray of that sample index of the
 * pixel's RNG stream ONLY IF sample == 0 (later samples depend on the path lengths before them).
 * prim_out / t_out: w*h each, row-major, -1 / -1.0f on miss. Host pointers. */
int b200rt_trace_primary(b200rt_scene* scene, const float* camera17, int width, int height, int sample, int spp_for_seed,
                         int* prim_out, float* t_out, const b200rt_render_options* opts_or_null, b200rt_stats* stats_or_null);

/* Per-pixel feature buffers for a denoiser (OIDN's "albedo" / "normal" auxiliary images; the reference feeds OIDN the beauty
 * alone, utils.cpp:144-196): k x k stratified camera rays per pixel over its footprint, mean diffuse colour of the closest hit's
 * material and mean geometric normal (not renormalised; misses contribute 0). k = 1: exactly b200rt_trace_primary's un-jittered ray.
 * 3 floats per pixel each, row 0 = bottom; either output may be NULL (not both). opts: flags select the layout (as trace_primary);
 * rank/world must be 0/1. Multi-device scene: computed on its first device. stats: rays = samples = w*h*k*k. */
int b200rt_render_aovs(b200rt_scene* scene, const float* camera17, int width, int height, int samples_per_axis,
                       float* albedo_rgb_out_or_null, float* normal_xyz_out_or_null,
                       const b200rt_render_options* opts_or_null, b200rt_stats* stats_or_null);

/* Replaces BVH::intersect / FlattenedBVH::intersect for a batch (source/bvh.cpp:62-65, flattened_bvh.cpp:10-58):
 * rays6 = {origin xyz, direction xyz}; extra8_or_null receives {point xyz, normal xyz, u, v} per ray. Host pointers.
 * any_hit != 0 returns 1/0 in prim_out (any triangle or sphere hit with t > 0) instead of the closest index. */
int b200rt_trace_rays(b200rt_scene* scene, const float* rays6, int n_rays, int any_hit,
                      int* prim_out, float* t_out, float* extra8_or_null, const b200rt_render_options* opts_or_null);

/* ---- device-pointer variants (the torch.distributed plumbing in bench.py / the multi-GPU host uses these) ------------
 * All run on `cuda_stream` (a cudaStream_t; NULL = legacy default stream) of the scene's device and do not synchronise
 * unless stats are requested. Tiles: the frame is cut into 16x16-pixel tiles, tile_id = ty * tiles_x + tx, owned by
 * rank tile_id % world; each rank fills a compact tile-major float4 buffer of b200rt_tiles_for_rank() * 256 pixels. */
int b200rt_tiles_for_rank(int width, int height, int rank, int world);
int b200rt_render_tiles_device(b200rt_scene* scene, const float* camera17, int width, int height, int spp, int max_bounces,
                               void* dev_tiles_rgba, const b200rt_render_options* opts_or_null, void* cuda_stream,
                               b200rt_stats* stats_or_null);
/* gathered: world consecutive per-rank tile buffers of tiles_per_rank_padded*256 float4 each (rank-major, as an
 * all-gather leaves them) -> row-major bottom-up RGBA image on the device */
int b200rt_untile_device(b200rt_scene* scene, const void* dev_gathered_tiles, int tiles_per_rank_padded, int world,
                         int width, int height, void* dev_image_rgba, void* cuda_stream);
/* As b200rt_untile_device, but for B200RT_FLAG_LINEAR_TILES tile buffers: dev_framebuffer_rgba_inout holds the incoming
 * framebuffer and receives `fb += final; fb = tone_map(fb)` (render_kernel.cpp:169-180) in place. */
int b200rt_untile_accumulate_device(b200rt_scene* scene, const void* dev_gathered_tiles, int tiles_per_rank_padded, int world,
                                    int width, int height, void* dev_framebuffer_rgba_inout, void* cuda_stream);
int b200rt_trace_primary_device(b200rt_scene* scene, const float* camera17, int width, int height, int sample, int spp_for_seed,
                                void* dev_prim, void* dev_t, const b200rt_render_options* opts_or_null, void* cuda_stream,
                                b200rt_stats* stats_or_null);
/* device-pointer variant of b200rt_render_aovs (w*h*3 floats each, either may be NULL, not both) */
int b200rt_render_aovs_device(b200rt_scene* scene, const float* camera17, int width, int height, int samples_per_axis,
                              void* dev_albedo_rgb_or_null, void* dev_normal_xyz_or_null,
                              const b200rt_render_options* opts_or_null, void* cuda_stream, b200rt_stats* stats_or_null);

/* device-pointer variant of b200rt_trace_rays (dev_extra8 may be NULL) */
int b200rt_trace_rays_device(b200rt_scene* scene, const void* dev_rays6, int n_rays, int any_hit, void* dev_prim, void* dev_t,
                             void* dev_extra8_or_null, const b200rt_render_options* opts_or_null, void* cuda_stream,
                             b200rt_stats* stats_or_null);

/* ---- output stage -------------------------------------------------------------------------------------------------------
 * The quantisation loop of write_image_png (source/image_io.cpp:165-182): out = (unsigned char)clamp(rgba * 255, 0, 255),
 * flip_y != 0 writes image row 0 (the bottom row) last, as stbi_flip_vertically_on_write does. 16 B in, 4 B out per
 * pixel: run it on the device right after a render and the frame leaves the GPU at a quarter of the bytes. */
int b200rt_quantise_rgba8(const float* image_rgba, int width, int height, int flip_y, unsigned char* out_rgba8);
int b200rt_quantise_rgba8_device(const void* dev_image_rgba, int width, int height, int flip_y, void* dev_out_rgba8, void* cuda_stream);

/* The denoise stage of main.cpp:118-120 (Utils::OIDN_denoise, source/utils.cpp:144-196: OIDN "RT" filter on the tone-mapped beauty
 * image alone, then out = blend * denoised + (1 - blend) * noisy, alpha 1). The reference does not ship OIDN's binaries or weights,
 * so there is nothing to be bit-compatible with: this is an edge-avoiding a-trous wavelet filter (5 passes, colour-guided) in the same
 * place — a functional stand-in, not a parity claim (DESIGN.md). channels: 3 (OIDN's float3 buffers) or 4 (Image). iterations <= 0
 * and sigma <= 0 or NaN select the defaults (5, 0.45); iterations above 8 are clamped to 8. in == out is allowed. Host pointers;
 * runs on the current device.
 * Non-finite pixels: a pixel with a NaN or +-Inf in R, G or B is missing data. It contributes to no neighbour, is left out of the
 * first pass's local-variance estimate, and is itself filtered from its finite neighbours without the colour term; its output is
 * the denoised value alone, whatever blend_factor. A pixel with no finite pixel within reach of any pass stays non-finite (an all-NaN
 * image stays NaN). The alpha channel is never inspected. Finite images are filtered exactly as if this rule did not exist. */
int b200rt_denoise(const float* image, int channels, int width, int height, float blend_factor, int iterations, float sigma, float* out);
/* b200rt_denoise with OIDN's auxiliary images as edge-stopping guides (w*h*3 floats each, either may be NULL; b200rt_render_aovs
 * computes them): a tap must also agree in normal direction and albedo to contribute. Both NULL: identical to b200rt_denoise, bit for bit. */
int b200rt_denoise_guided(const float* image, int channels, const float* albedo_rgb_or_null, const float* normal_xyz_or_null,
                          int width, int height, float blend_factor, int iterations, float sigma, float* out);

const char* b200rt_last_error(void);
const char* b200rt_version(void);

#ifdef __cplusplus
}
#endif
#endif
