// Launchers of the sm_100a kernels (kernels.cu). Host code only sees these.
#pragma once
#include <vector>

#include <cuda_runtime.h>

#include "../../include/b200rt.h"
#include "bvh_build.h"
#include "device_types.h"

namespace b200rt {

// Which traversal a launch uses. Incoherent rays (the integrators, ray batches) default to the 8-ary quantised BVH: fewer
// dependent fetches and bytes per ray. Coherent camera rays (k_primary) default to the binary layout: its exact
// near-first order with per-entry distance culling does less work per ray when a whole warp walks the same nodes
// (C2: 5.9 vs 3.8 Grays/s, C5 primary: 2.0 vs 1.1 Grays/s). B200RT_FLAG_BVH2 / B200RT_FLAG_BVH8 force one or the other.
inline int traversal_layout(const SceneDev& S, int flags, bool coherent = false)
{
    const bool binary = (flags & (B200RT_FLAG_BVH2 | B200RT_FLAG_DIAG_SLABS)) || (coherent && !(flags & B200RT_FLAG_BVH8));
    if (S.has_wide && !binary) return 2;                                                  // TL_WIDE
    return (S.has_diag && (flags & B200RT_FLAG_DIAG_SLABS)) ? 1 : 0;                      // TL_DIAG : TL_AXIS
}

// SM count of the current device (cached per device id)
int current_sm_count();
// B200RT_TILE_SKEW (device_types.h tile_xy), read once per process
int tile_skew();

cudaError_t launch_megakernel(const SceneDev& S, const RenderParams& P, const float4* fb_in_rowmajor, float4* out_tiles,
                              unsigned int* work_counter, unsigned long long* ray_counter, cudaStream_t stream);
cudaError_t launch_primary(const SceneDev& S, const RenderParams& P, int sample, int* prim_out, float* t_out, cudaStream_t stream);
// feature buffers (k x k stratified camera rays per pixel): mean albedo and geometric normal, 3 floats per pixel each, either may be null
cudaError_t launch_aov(const SceneDev& S, const RenderParams& P, int k, float* albedo_out, float* normal_out, cudaStream_t stream);
cudaError_t launch_trace_rays(const SceneDev& S, const float* rays6, int n, int any_hit, int flags, int* prim_out, float* t_out,
                              float* extra8, cudaStream_t stream);
cudaError_t launch_untile(const float4* tiles, int tiles_per_rank_padded, int world, int only_rank, int w, int h, float4* image,
                          cudaStream_t stream);

cudaError_t launch_untile_accumulate(const float4* tiles, int tiles_per_rank_padded, int world, int w, int h, float4* image, cudaStream_t stream);
cudaError_t launch_fill_f4(float4* p, size_t n, float4 v, cudaStream_t stream);
cudaError_t launch_fill_f32(float* p, size_t n, float v, cudaStream_t stream);
cudaError_t launch_env_cdf_search(const SceneDev& S, const float* values, int n, int* xy, cudaStream_t stream);
cudaError_t launch_rng_stream(int x, int y, int spp, int n, uint32_t* state_out, float* floats_out, cudaStream_t stream);
cudaError_t launch_quantise_rgba8(const float4* image, int w, int h, int flip_y, void* out_rgba8, cudaStream_t stream);

// output stage: edge-avoiding a-trous denoiser (denoise.cu); d_albedo / d_normal: optional w*h*3 guides (both null: colour only)
cudaError_t launch_denoise(const float* d_in, int channels, const float* d_albedo, const float* d_normal, int w, int h, int iterations,
                           float sigma, float blend, float* d_tmp, float* d_out, cudaStream_t stream);

// K5 env tables (env_tables.cu)
cudaError_t launch_env_expand_rgb(const float* rgb, size_t n, float4* rgba, cudaStream_t stream);
cudaError_t launch_env_luminance(const float4* env, size_t n, float* lum, cudaStream_t stream);
cudaError_t launch_env_cdf_serial(const float* lum, size_t n, float* cdf, cudaStream_t stream);
cudaError_t launch_env_row_cdf(const float* cdf, int w, int h, float* row, cudaStream_t stream);
cudaError_t build_env_cdf_guide(const float* cdf, size_t n, float total, int n_buckets, unsigned int* guide, float* scale_out, int* built_out, cudaStream_t stream);
cudaError_t build_env_alias_device(const float* lum, size_t n, float2* table, double* total_host, cudaStream_t stream);

// B200RT_FLAG_TIME_INLINE: every trace / shade launch of a frame bracketed by CUDA events on its own group stream, nothing
// serialised or synchronised while the frame runs; read back after the frame has finished (wavefront_timeline_summary)
struct WfTimeline
{
    struct Launch { int group; size_t e0, e1, e2; };      // events: trace start, trace end = shade start, shade end
    std::vector<cudaEvent_t> pool;
    size_t used = 0;
    std::vector<Launch> launches;
    std::vector<Launch> tails;                            // barrier-free tail launches (e0 .. e1; e2 unused)
    cudaEvent_t origin = nullptr;                         // recorded on the caller's stream at the fork
    cudaEvent_t take();
    void reset() { used = 0; launches.clear(); tails.clear(); }
    void destroy();
};
// sums (ms) and launch counts of the recorded frame, and the length of the union of the trace kernels' intervals: the time during
// which at least one trace kernel was running. The frame must have completed (stream synchronised).
struct WfTimelineSummary { double trace_ms, shade_ms, trace_union_ms, tail_ms; int trace_launches, shade_launches, tail_launches; };
cudaError_t wavefront_timeline_summary(const WfTimeline& tl, WfTimelineSummary* out);

// wavefront integrator (wavefront.cu): runs the whole frame for this rank's tiles as n_groups independent interleaved
// tile groups, each on its own stream; `stream` is forked from and joined back into
cudaError_t run_wavefront(const SceneDev& S, const RenderParams& P, const WfGroup* groups, int n_groups, const float4* fb_in_rowmajor,
                          float4* out_tiles, cudaStream_t stream, cudaEvent_t fork_event, int* launches_out, double* kernel_times4 = nullptr,
                          unsigned int* unfinished_out = nullptr, WfTimeline* timeline = nullptr);
cudaError_t wavefront_sum_rays(const WfGroup* groups, int n_groups, unsigned long long* total, cudaStream_t stream);

// barrier-free tail of a pass-synchronous frame (persist.cu): finishes the group's unfinished slots in one launch
cudaError_t launch_wavefront_tail(const SceneDev& S, const RenderParams& P, const WfBuffers& B, int max_ctas, const float4* fb_in_rowmajor,
                                  float4* out_tiles, cudaStream_t stream);
int wavefront_tail_max_ctas();

// persistent integrator (persist.cu): one launch per frame, every warp its own wavefront machine
int persistent_grid();
int persistent_slots(int grid);
cudaError_t run_persistent(const SceneDev& S, const RenderParams& P, const WfBuffers& B, int grid, const float4* fb_in_rowmajor,
                           float4* out_tiles, cudaStream_t stream);

// refit of a resident tree to new vertices of the same triangles (refit.cu; b200rt_scene_update_triangles)
// misc[0] = max |coord| as float bits, misc[1] = 1 when a coordinate is NaN or +-Inf (misc: 2 words, zeroed here)
cudaError_t refit_extent(const float* tri9, int n_tri, unsigned int* misc, cudaStream_t stream);
// the nodes of each layout grouped by tree level, by a breadth-first walk from record 0: level k is idx[level[k] .. level[k + 1]).
// Synchronises `stream`. cudaErrorInvalidValue: the records do not form one tree rooted at record 0.
cudaError_t refit_levels(const WideNode* wide, int n_wide, const AxisNode* axis, int n_axis, int* wide_idx, int* axis_idx, int* counter,
                         std::vector<int>& wide_level, std::vector<int>& axis_level, cudaStream_t stream);
size_t refit_sah_scratch_doubles();
struct RefitArgs
{
    const float* tri9;                     // new vertices, original triangle order, on this device
    float4* tris; WideNode* wide; AxisNode* axis; DiagNode* diag;        // the resident arrays (diag: null = not refitted)
    const int* wide_idx; const int* axis_idx;
    const std::vector<int>* wide_level; const std::vector<int>* axis_level;
    float4* wide_box; float4* axis_box;    // per-node exact boxes: 2 float4 per wide node, 4 per binary record
    int n_tri, n_axis;
    float abs_pad;
    int* overflow;                         // set when a quantised box does not fit its node's grid
    double* sah;                           // refit_sah_scratch_doubles(); the SAH cost lands in the last one
};
// triangle stream, then every level of both layouts deepest first, then the SAH cost; *launches = kernels launched
cudaError_t refit_tree(const RefitArgs& args, cudaStream_t stream, int* launches);
// the SAH cost of n_axis > 0 binary records (sah_cost_of's formula, fixed summation order) into sah[refit_sah_scratch_doubles() - 1]; 2 launches
cudaError_t refit_sah(const AxisNode* axis, int n_axis, double* sah, cudaStream_t stream);

} // namespace b200rt
