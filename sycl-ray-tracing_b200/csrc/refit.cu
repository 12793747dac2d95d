// Refit of a resident BVH to new vertex positions (b200rt_scene_update_triangles): the topology stays, every box is recomputed
// bottom-up from the new vertices.
//   1. extent pass: max |coord| (the abs_pad both builders derive from it) and a non-finite flag         (rf_extent)
//   2. the leaf-ordered triangle stream, {a, b - a, c - a} of the triangle each slot already holds     (rf_triangles)
//   3. one launch per tree level, deepest first, for each layout: a node's exact (unpadded) box goes to a per-node scratch array,
//      and the node pads its children's exact boxes once, exactly as the builders do                  (rf_wide_level, rf_axis_level)
//   4. the SAH cost of the refitted binary records, sah_cost_of's formula, in double                   (rf_sah_partial, rf_sah_final)
// Level lists come from a breadth-first walk from record 0 (rf_bfs_*): record order is not a topological order (append_top_level
// moves the old root to the end of both arrays).
#include <algorithm>
#include <cfloat>
#include <cstdint>
#include <vector>

#include <cuda_runtime.h>

#include "bvh_build.h"
#include "bvh_emit.cuh"
#include "kernels.h"

namespace b200rt {
namespace {

constexpr int kRefitBlock = 128;
constexpr int kSahBlocks = 256, kSahThreads = 256;

__device__ __forceinline__ void grow(float* lo, float* hi, const float* p)
{
    for (int a = 0; a < 3; a++) { lo[a] = fminf(lo[a], p[a]); hi[a] = fmaxf(hi[a], p[a]); }
}

// ---- 1. extent ------------------------------------------------------------------------------------------------------------------
// misc[0]: max |coord| as float bits (non-negative floats order like their bits), misc[1]: 1 when some coordinate is NaN or +-Inf
__global__ void rf_extent(const float* __restrict__ tri9, size_t n_coords, unsigned int* misc)
{
    float am = 0.0f;
    int bad = 0;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n_coords; i += (size_t)gridDim.x * blockDim.x)
    {
        const float v = tri9[i];
        if (!isfinite(v)) bad = 1; else am = fmaxf(am, fabsf(v));
    }
    for (int o = 16; o > 0; o >>= 1) { am = fmaxf(am, __shfl_xor_sync(0xffffffffu, am, o)); bad |= __shfl_xor_sync(0xffffffffu, bad, o); }
    if ((threadIdx.x & 31) == 0)
    {
        atomicMax(&misc[0], __float_as_uint(am));
        if (bad) atomicOr(&misc[1], 1u);
    }
}

// ---- 2. triangle stream -----------------------------------------------------------------------------------------------------------
__global__ void rf_triangles(const float* __restrict__ tri9, float4* tris, int n)
{
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    emit_triangle(tri9, __float_as_int(tris[3 * (size_t)j].w), tris + 3 * (size_t)j);
}

// ---- level lists ----------------------------------------------------------------------------------------------------------------
// idx[begin, end) is one level; its children are appended behind `end` (count in *n_next)
__global__ void rf_bfs_wide(const WideNode* nodes, int* idx, int begin, int end, int* n_next)
{
    const int k = begin + blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= end) return;
    const WideNode& w = nodes[idx[k]];
    const int n_inner = __popc((unsigned)w.imask);
    if (!n_inner) return;
    const int at = end + atomicAdd(n_next, n_inner);
    for (int i = 0; i < n_inner; i++) idx[at + i] = (int)w.child_base + i;
}

__global__ void rf_bfs_axis(const AxisNode* axis, int* idx, int begin, int end, int* n_next)
{
    const int k = begin + blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= end) return;
    const AxisNode& r = axis[idx[k]];
    if (r.l_ref >= 0) idx[end + atomicAdd(n_next, 1)] = r.l_ref;
    if (r.r_ref >= 0) idx[end + atomicAdd(n_next, 1)] = r.r_ref;
}

// ---- 3. refit, one level per launch --------------------------------------------------------------------------------------------------
// exact box of the triangles in slots [first, first + count) of the stream, from the input vertices (never from a + e1: it does not
// round back to b)
__device__ __forceinline__ void leaf_box(const float4* tris, const float* tri9, int first, int count, float* lo, float* hi)
{
    for (int i = 0; i < count; i++)
    {
        const float* p = tri9 + 9 * (size_t)__float_as_int(tris[3 * (size_t)(first + i)].w);
        grow(lo, hi, p); grow(lo, hi, p + 3); grow(lo, hi, p + 6);
    }
}

// wide node idx[k]: quantised child boxes from the children's exact boxes (inner: box[child], leaf: its triangles), padded once;
// box[node] = the union of its children's exact boxes (2 float4: lo, hi)
__global__ void __launch_bounds__(kRefitBlock) rf_wide_level(WideNode* nodes, const int* __restrict__ idx, int n, const float4* __restrict__ tris,
                                                            const float* __restrict__ tri9, float4* box, float abs_pad, int* overflow)
{
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const int me = idx[k];
    WideNode node = nodes[me];
    float klo[8][3], khi[8][3];
    float ulo[3] = { FLT_MAX, FLT_MAX, FLT_MAX }, uhi[3] = { -FLT_MAX, -FLT_MAX, -FLT_MAX };
    unsigned used = 0;
    int inner_rank = 0, tri_at = (int)node.tri_base;
    for (int s = 0; s < 8; s++)
    {
        float lo[3] = { FLT_MAX, FLT_MAX, FLT_MAX }, hi[3] = { -FLT_MAX, -FLT_MAX, -FLT_MAX };
        const unsigned m = (node.valid24 >> (3 * s)) & 7u;
        if ((node.imask >> s) & 1)
        {
            const int c = (int)node.child_base + inner_rank++;
            const float4 cl = box[2 * (size_t)c], ch = box[2 * (size_t)c + 1];
            lo[0] = cl.x; lo[1] = cl.y; lo[2] = cl.z; hi[0] = ch.x; hi[1] = ch.y; hi[2] = ch.z;
        }
        else if (m)
        {
            const int cnt = __popc(m);
            leaf_box(tris, tri9, tri_at, cnt, lo, hi);
            tri_at += cnt;
        }
        else continue;
        used |= 1u << s;
        for (int a = 0; a < 3; a++)
        {
            const float pad = box_pad_dev(lo[a], hi[a], abs_pad);
            klo[s][a] = lo[a] - pad; khi[s][a] = hi[a] + pad;
        }
        grow(ulo, uhi, lo); grow(ulo, uhi, hi);
    }
    wide_quantise(node, klo, khi, used, overflow);
    nodes[me] = node;
    box[2 * (size_t)me] = make_float4(ulo[0], ulo[1], ulo[2], 0.0f);
    box[2 * (size_t)me + 1] = make_float4(uhi[0], uhi[1], uhi[2], 0.0f);
}

// exact 7-plane volume of a subtree: the 3 axis slabs and the 4 diagonal distances (4 float4: lo, hi, near, far)
struct Slabs7 { float lo[3], hi[3], dnear[4], dfar[4]; };

__device__ __forceinline__ void slabs_reset(Slabs7& s)
{
    for (int a = 0; a < 3; a++) { s.lo[a] = INFINITY; s.hi[a] = -INFINITY; }
    for (int k = 0; k < 4; k++) { s.dnear[k] = INFINITY; s.dfar[k] = -INFINITY; }
}

// Slabs::grow_point of bvh_build.cpp: the diagonal distance exact in double, rounded outward to float
__device__ __forceinline__ void slabs_grow_point(Slabs7& s, const float* p)
{
    grow(s.lo, s.hi, p);
    for (int k = 0; k < 4; k++)
    {
        double d;
        switch (k)
        {
        case 0: d = (double)p[0] + (double)p[1] + (double)p[2]; break;
        case 1: d = -(double)p[0] + (double)p[1] + (double)p[2]; break;
        case 2: d = -(double)p[0] - (double)p[1] + (double)p[2]; break;
        default: d = (double)p[0] - (double)p[1] + (double)p[2]; break;
        }
        const float f = (float)d;
        const float fl = ((double)f > d) ? nextafterf(f, -INFINITY) : f;
        const float fh = ((double)f < d) ? nextafterf(f, INFINITY) : f;
        s.dnear[k] = fminf(s.dnear[k], fl);
        s.dfar[k] = fmaxf(s.dfar[k], fh);
    }
}

__device__ __forceinline__ void slabs_grow(Slabs7& s, const Slabs7& o)
{
    for (int a = 0; a < 3; a++) { s.lo[a] = fminf(s.lo[a], o.lo[a]); s.hi[a] = fmaxf(s.hi[a], o.hi[a]); }
    for (int k = 0; k < 4; k++) { s.dnear[k] = fminf(s.dnear[k], o.dnear[k]); s.dfar[k] = fmaxf(s.dfar[k], o.dfar[k]); }
}

// binary record idx[k]: both children's axis slabs (and diagonal slabs when `diag` is given) from their exact volumes, padded once as
// Flattener::store_child pads them; an empty leaf keeps its inverted, never-hit volume. box[record] = the union of both children.
__global__ void __launch_bounds__(kRefitBlock) rf_axis_level(AxisNode* axis, DiagNode* diag, const int* __restrict__ idx, int n,
                                                            const float4* __restrict__ tris, const float* __restrict__ tri9, float4* box, float abs_pad)
{
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const int me = idx[k];
    AxisNode an = axis[me];
    DiagNode dn;
    if (diag) dn = diag[me];
    Slabs7 u;
    slabs_reset(u);
    for (int side = 0; side < 2; side++)
    {
        const int ref = side ? an.r_ref : an.l_ref;
        float* lo = side ? an.r_lo : an.l_lo; float* hi = side ? an.r_hi : an.l_hi;
        float* dnear = side ? dn.r_near : dn.l_near; float* dfar = side ? dn.r_far : dn.l_far;
        Slabs7 s;
        slabs_reset(s);
        if (ref >= 0)
        {
            const float4* b = box + 4 * (size_t)ref;
            const float4 b0 = b[0], b1 = b[1], b2 = b[2], b3 = b[3];
            s.lo[0] = b0.x; s.lo[1] = b0.y; s.lo[2] = b0.z; s.hi[0] = b1.x; s.hi[1] = b1.y; s.hi[2] = b1.z;
            s.dnear[0] = b2.x; s.dnear[1] = b2.y; s.dnear[2] = b2.z; s.dnear[3] = b2.w;
            s.dfar[0] = b3.x; s.dfar[1] = b3.y; s.dfar[2] = b3.z; s.dfar[3] = b3.w;
        }
        else
        {
            const int first = (~ref) >> 4, count = (~ref) & 15;
            if (count == 0)
            {
                for (int a = 0; a < 3; a++) { lo[a] = INFINITY; hi[a] = -INFINITY; }
                for (int q = 0; q < 4; q++) { dnear[q] = INFINITY; dfar[q] = -INFINITY; }
                continue;
            }
            for (int i = 0; i < count; i++)
            {
                const float* p = tri9 + 9 * (size_t)__float_as_int(tris[3 * (size_t)(first + i)].w);
                slabs_grow_point(s, p); slabs_grow_point(s, p + 3); slabs_grow_point(s, p + 6);
            }
        }
        for (int a = 0; a < 3; a++)
        {
            const float pad = box_pad_dev(s.lo[a], s.hi[a], abs_pad);
            lo[a] = s.lo[a] - pad; hi[a] = s.hi[a] + pad;
        }
        for (int q = 0; q < 4; q++)
        {
            const float pad = 1e-5f * fmaxf(fabsf(s.dnear[q]), fabsf(s.dfar[q])) + 2.0f * abs_pad;
            dnear[q] = s.dnear[q] - pad; dfar[q] = s.dfar[q] + pad;
        }
        slabs_grow(u, s);
    }
    axis[me] = an;
    if (diag) diag[me] = dn;
    float4* b = box + 4 * (size_t)me;
    b[0] = make_float4(u.lo[0], u.lo[1], u.lo[2], 0.0f);
    b[1] = make_float4(u.hi[0], u.hi[1], u.hi[2], 0.0f);
    b[2] = make_float4(u.dnear[0], u.dnear[1], u.dnear[2], u.dnear[3]);
    b[3] = make_float4(u.dfar[0], u.dfar[1], u.dfar[2], u.dfar[3]);
}

// ---- 4. SAH cost (sah_cost_of in bvh_build.cpp) ----------------------------------------------------------------------------------------
__device__ __forceinline__ double half_area_d(const float* lo, const float* hi)
{
    const double dx = (double)hi[0] - lo[0], dy = (double)hi[1] - lo[1], dz = (double)hi[2] - lo[2];
    return (dx < 0 || dy < 0 || dz < 0) ? 0.0 : dx * dy + dy * dz + dz * dx;
}

__device__ __forceinline__ double block_sum(double v, double* sh)
{
    sh[threadIdx.x] = v;
    __syncthreads();
    for (int o = kSahThreads / 2; o > 0; o >>= 1)
    {
        if ((int)threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
        __syncthreads();
    }
    return sh[0];
}

// fixed grid and fixed summation order: the same records give the same bits
__global__ void __launch_bounds__(kSahThreads) rf_sah_partial(const AxisNode* axis, int n, double* partial)
{
    __shared__ double sh[kSahThreads];
    const AxisNode& r = axis[0];
    float lo[3], hi[3];
    for (int a = 0; a < 3; a++) { lo[a] = fminf(r.l_lo[a], r.r_lo[a]); hi[a] = fmaxf(r.l_hi[a], r.r_hi[a]); }
    const double root_area = fmax(1e-30, half_area_d(lo, hi));
    double acc = 0.0;
    for (int i = blockIdx.x * kSahThreads + threadIdx.x; i < n; i += kSahBlocks * kSahThreads)
    {
        const AxisNode& x = axis[i];
        const double al = half_area_d(x.l_lo, x.l_hi) / root_area, ar = half_area_d(x.r_lo, x.r_hi) / root_area;
        acc += x.l_ref >= 0 ? al : al * x.l_count;
        acc += x.r_ref >= 0 ? ar : ar * x.r_count;
    }
    const double s = block_sum(acc, sh);
    if (threadIdx.x == 0) partial[blockIdx.x] = s;
}

__global__ void __launch_bounds__(kSahThreads) rf_sah_final(double* partial)
{
    __shared__ double sh[kSahThreads];
    const double s = block_sum(partial[threadIdx.x], sh);
    if (threadIdx.x == 0) partial[kSahBlocks] = 1.0 + s;
}

static_assert(kSahBlocks == kSahThreads, "rf_sah_final sums one partial per thread");

int blocks_for(size_t n, int tb) { return (int)((n + tb - 1) / tb); }

} // namespace

size_t refit_sah_scratch_doubles() { return kSahBlocks + 1; }

cudaError_t refit_extent(const float* tri9, int n_tri, unsigned int* misc, cudaStream_t st)
{
    cudaError_t e = cudaMemsetAsync(misc, 0, 2 * sizeof(unsigned int), st);
    if (e != cudaSuccess) return e;
    const size_t n = 9 * (size_t)n_tri;
    const int grid = (int)std::min<size_t>(4 * (size_t)current_sm_count(), (size_t)blocks_for(n, 256));
    if (grid > 0) rf_extent<<<grid, 256, 0, st>>>(tri9, n, misc);
    return cudaGetLastError();
}

cudaError_t refit_levels(const WideNode* wide, int n_wide, const AxisNode* axis, int n_axis, int* wide_idx, int* axis_idx, int* counter,
                         std::vector<int>& wide_level, std::vector<int>& axis_level, cudaStream_t st)
{
    for (int layout = 0; layout < 2; layout++)
    {
        const int n_nodes = layout ? n_axis : n_wide;
        int* idx = layout ? axis_idx : wide_idx;
        std::vector<int>& level = layout ? axis_level : wide_level;
        level.assign(1, 0);
        if (!n_nodes) continue;
        const int zero = 0;
        cudaError_t e = cudaMemcpyAsync(idx, &zero, sizeof(int), cudaMemcpyHostToDevice, st);
        int begin = 0, end = 1;
        while (e == cudaSuccess && begin < end)
        {
            level.push_back(end);
            int next = 0;
            e = cudaMemsetAsync(counter, 0, sizeof(int), st);
            if (e != cudaSuccess) break;
            if (layout) rf_bfs_axis<<<blocks_for(end - begin, 256), 256, 0, st>>>(axis, idx, begin, end, counter);
            else rf_bfs_wide<<<blocks_for(end - begin, 256), 256, 0, st>>>(wide, idx, begin, end, counter);
            if ((e = cudaMemcpyAsync(&next, counter, sizeof(int), cudaMemcpyDeviceToHost, st)) == cudaSuccess) e = cudaStreamSynchronize(st);
            if (e != cudaSuccess) break;
            if (next > n_nodes - end || (int)level.size() > kMaxTraversalDepth + 8) return cudaErrorInvalidValue;   // not a tree
            begin = end; end += next;
        }
        if (e != cudaSuccess) return e;
        if (end != n_nodes) return cudaErrorInvalidValue;      // some record is not reachable from record 0
    }
    return cudaSuccess;
}

cudaError_t refit_tree(const RefitArgs& R, cudaStream_t st, int* launches)
{
    const int n_tri = R.n_tri;
    *launches = 0;
    if (n_tri > 0) { rf_triangles<<<blocks_for((size_t)n_tri, 256), 256, 0, st>>>(R.tri9, R.tris, n_tri); ++*launches; }
    for (int l = (int)R.wide_level->size() - 2; l >= 0; l--)
    {
        const int b = (*R.wide_level)[(size_t)l], n = (*R.wide_level)[(size_t)l + 1] - b;
        rf_wide_level<<<blocks_for((size_t)n, kRefitBlock), kRefitBlock, 0, st>>>(R.wide, R.wide_idx + b, n, R.tris, R.tri9, R.wide_box, R.abs_pad, R.overflow);
        ++*launches;
    }
    for (int l = (int)R.axis_level->size() - 2; l >= 0; l--)
    {
        const int b = (*R.axis_level)[(size_t)l], n = (*R.axis_level)[(size_t)l + 1] - b;
        rf_axis_level<<<blocks_for((size_t)n, kRefitBlock), kRefitBlock, 0, st>>>(R.axis, R.diag, R.axis_idx + b, n, R.tris, R.tri9, R.axis_box, R.abs_pad);
        ++*launches;
    }
    if (R.n_axis > 0)
    {
        rf_sah_partial<<<kSahBlocks, kSahThreads, 0, st>>>(R.axis, R.n_axis, R.sah);
        rf_sah_final<<<1, kSahThreads, 0, st>>>(R.sah);
        *launches += 2;
    }
    return cudaGetLastError();
}

} // namespace b200rt
