// Host-side builder for the re-laid-out FlattenedBVH (layout documented in include/b200rt.h).
// Replaces BVH::BVH / OctreeNode::insert / compute_volume / flatten of the reference
// (source/bvh.cpp:19-60, include/bvh.h:55-125, :211-250): only the closest-hit RESULT is contractual, not the tree
// shape, so this is a binned-SAH binary BVH whose nodes carry the reference's 7-plane Kay-Kajiya slab volumes
// (include/bounding_volume.h:9-127, plane normals source/bvh.cpp:8-16).
#pragma once
#include <cstdint>
#include <functional>
#include <string>
#include <vector>

#include <cuda_runtime.h>

#include "../../include/b200rt.h"

namespace b200rt {

constexpr int kMaxTraversalDepth = 60;   // the device stack holds 64 entries

struct alignas(64) AxisNode
{
    float l_lo[3], l_hi[3], r_lo[3], r_hi[3];
    int l_ref, r_ref, l_count, r_count;
};
static_assert(sizeof(AxisNode) == 64, "axis record is one 64-byte line");

struct alignas(64) DiagNode
{
    float l_near[4], l_far[4], r_near[4], r_far[4];
};
static_assert(sizeof(DiagNode) == 64, "diag record is one 64-byte line");

struct alignas(16) LeafTriangle
{
    float a[3]; int prim;      // vertex a + original triangle index
    float e1[3]; float pad1;   // b - a   (same float subtraction the reference does per test, triangle.h:21)
    float e2[3]; float pad2;   // c - a   (triangle.h:22)
};
static_assert(sizeof(LeafTriangle) == 48, "three float4 per triangle");

// node of the 8-ary quantised BVH (device twin and the plane decoding: csrc/pt_device.cuh, "wide BVH")
struct alignas(16) WideNode
{
    float p[3];                 // frame origin
    uint8_t e[3];               // per-axis cell size 2^(e - 127)
    uint8_t imask;              // bit s set: slot s holds an inner child
    uint32_t child_base;        // node index of the first inner child (inner children are contiguous, in slot order)
    uint32_t tri_base;          // slot of the first triangle of this node's leaf children (contiguous, in slot order)
    uint32_t valid24;           // bit 3s + i: slot s is a leaf child with a triangle i; triangles are stored compactly in that bit order
    uint32_t spare;
    uint8_t lox[8], loy[8], loz[8], hix[8], hiy[8], hiz[8];   // quantised child boxes, one byte per plane
};
static_assert(sizeof(WideNode) == 80, "five float4 per wide node");

// plane byte -> grid value: the float with bits 0x43000000 | q << 16 (128 + q below 128, 2q from 128 on)
inline int wide_grid_value(int q) { return q < 128 ? 128 + q : 2 * q; }
constexpr int kWideMaxLeaf = 3;          // a leaf child's triangle count is unary-coded in 3 bits

struct FlatBVH
{
    std::vector<WideNode> wide;
    std::vector<AxisNode> axis;
    std::vector<DiagNode> diag;
    std::vector<LeafTriangle> tris;
    b200rt_bvh_info info{};
};

// the 4 diagonal plane normals WITHOUT the sqrt(3)/3 factor: distances along (+-1, +-1, 1) give the same slab
// intersection parameters t as the reference's normalised planes (both numerator and denominator scale alike)
inline float diag_dist(int k, float x, float y, float z)
{
    switch (k)
    {
    case 0: return (x + y) + z;
    case 1: return (-x + y) + z;
    case 2: return (-x - y) + z;
    default: return (x - y) + z;
    }
}

void build_flat_bvh(const float* tri9, int n_tri, const b200rt_bvh_options& opts, FlatBVH& out);
int check_flat_bvh(const FlatBVH& bvh, const float* tri9, int n_tri);
double sah_cost_of(const FlatBVH& bvh);
// Triangles kept out of the tree (the device builder's outsized ones) become leaf children of extra top-level nodes in front of both
// layouts' roots (bvh_build.cpp). From record 0 of each layout (w0, a0), the existing record counts, the extra triangles' vertices
// (extra9: 9 floats each; their stream slots start at first_slot) and the tree's abs_pad: out.wide[0] / out.axis[0] replace record 0,
// out.wide[1 + j] / out.axis[1 + j] become records n_wide + j / n_axis + j (the old root first). info's counts and depths follow.
struct TopLevel { std::vector<WideNode> wide; std::vector<AxisNode> axis; };
inline int top_level_wide(int n_extra) { return (n_extra + 7 * kWideMaxLeaf - 1) / (7 * kWideMaxLeaf); }
inline int top_level_axis(int n_extra) { return (n_extra + 14) / 15; }
void make_top_level(const WideNode& w0, const AxisNode& a0, size_t n_wide, size_t n_axis, size_t first_slot, const float* extra9, int n_extra,
                    float abs_pad, TopLevel& out, b200rt_bvh_info& info);

// ---- device builder (bvh_build_gpu.cu): 0 = ok, 1 = CUDA error, 2 = input outside what it handles (err says why) ----------------------
// Where a device build writes its tree: arrays the caller owns and allocates when the build asks, once the sizes are known (again
// for a second attempt, which replaces the first one's). wide_and_tris: n_wide WideNodes (5 float4 each), then the n_tri-record
// triangle stream (3 float4 each) in the same allocation; axis: n_axis binary records.
struct DeviceTree { float4* wide_and_tris = nullptr; AxisNode* axis = nullptr; };
using DeviceTreeAlloc = std::function<cudaError_t(size_t n_wide, size_t n_axis, DeviceTree& out)>;
struct DeviceBuildCounts { int launches = 0; unsigned long long h2d_bytes = 0, d2h_bytes = 0; };   // library sorts and scans count as one launch each
// Builds over d_tri9 (device memory of the current device) on stream st, into the caller's arrays; info gets everything but
// build_seconds and sah_cost. Clustering first; an input it gives up on gets the Morton radix tree. Synchronises st.
int build_bvh_device(const float* d_tri9, int n_tri, cudaStream_t st, const DeviceTreeAlloc& alloc, b200rt_bvh_info& info,
                     DeviceBuildCounts& counts, std::string& err);
// the same build from host vertices into a host FlatBVH: upload, build_bvh_device, download
int build_flat_bvh_device(const float* tri9_host, int n_tri, int device, FlatBVH& out, std::string& err);
// slot_of_prim[prim of stream record j] = j for the n_tri records of a triangle stream
cudaError_t launch_slot_of_prim(const float4* tris, int n_tri, int* slot_of_prim, cudaStream_t st);

} // namespace b200rt
