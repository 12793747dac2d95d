// BVH construction on the device (sm_100a): replaces BVH::BVH / OctreeNode::insert / compute_volume / flatten of the
// reference (source/bvh.cpp:19-60, include/bvh.h:55-125, :211-250) for callers that cannot afford the host builder
// (SURVEY §8f rank 1: at 20 M triangles the host SAH build is ~13 s, the reference's own octree insert is sequential).
// Only the closest-hit RESULT is contractual (SURVEY a15), not the tree shape, so this is a linear BVH:
//   1. per-triangle boxes, scene bounds                                   (lb_bounds)
//   2. 63-bit Morton codes of the box centres, radix sort                 (lb_morton, cub::DeviceRadixSort — library call, one-shot setup)
//   3. binary tree over the sorted triangles by PARALLEL LOCALLY-ORDERED CLUSTERING (pl_*; Meister & Bittner, "Parallel locally-ordered
//      clustering for bounding volume hierarchy construction", TVCG 2018): every cluster looks 16 places left and right along the
//      Morton curve for the neighbour whose merged box has the smallest surface area; mutual nearest neighbours merge; repeat
//      (~30 rounds). A surface-area-driven agglomerative build: round 1 built the radix tree of the Morton codes instead (Karras 2012,
//      lb_tree + lb_fit), whose splits ignore surface area — path tracing was 8-13 % and coherent camera rays 57 % slower on its
//      trees than on the host builder's binned-SAH ones. The radix tree remains the fallback for inputs that clustering refuses
//      (more than 512 rounds, or a tree deeper than the traversal stack)
//   4. the clustered tree is laid out depth-first (pl_layout): every subtree covers a contiguous range of the triangle order
//   5. subtrees of <= 3 triangles become leaves; level-by-level collapse into the 8-ary layout: every wide node opens its
//      largest children until it has 8, assigns them to octant slots     (lw_expand, lw_link; prefix sums give child_base / tri_base)
//   6. emit: quantised 80-byte wide nodes + the leaf-ordered triangle stream (lw_emit), binary two-children records (lb_emit)
// Outsized triangles (box diagonal > 1/4 of the scene's: a ground quad under a mesh) would drag every ancestor box of their
// Morton leaf out to the whole scene; up to 45 of them are kept out of the tree and hung, as leaf children, under one to
// three extra top-level nodes in front of the tree's root (make_top_level: the host works them out from record 0 of each layout and
// the outsized triangles' vertices, and writes them back).
// The build reads vertices already on the device and writes into arrays its caller owns (build_bvh_device): a resident scene rebuilds
// its tree in place with it, and b200rt_bvh_build_device is upload, build, download (build_flat_bvh_device).
// Output is the same FlatBVH the host builder produces (b200rt_bvh_check validates either), except that it carries no
// diagonal slabs (has_diag_slabs = 0: the 7-plane ablation needs the host builder).
#include <algorithm>
#include <cfloat>
#include <chrono>
#include <cstdint>
#include <cstring>
#include <string>
#include <vector>

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <cuda_runtime.h>

#include "bvh_build.h"
#include "bvh_emit.cuh"

namespace b200rt {
namespace {

constexpr int kLeafBit = 0x40000000;        // child reference of the radix tree: index | kLeafBit = sorted triangle position

struct DevArrays
{
    const float* tri9;
    float4 *plo, *phi;                       // per triangle box
    unsigned long long *keys, *keys_alt;
    int *vals, *vals_alt;                    // sorted position -> triangle index
    int *left, *right, *first, *last, *parent_node, *parent_leaf;
    float4 *nlo, *nhi;                       // per internal node box
    unsigned int* visits;
    int* scene;                              // ordered ints: [0..5] centre-bounds min xyz / max xyz, [6] max |coord|, [8..13] scene box min / max; [14] = outsized count
    int segregate;                           // 1: outsized triangles get the largest sort key and stay out of the tree
    int n;
    int leaf_max;                            // subtrees of at most this many triangles (<= kWideMaxLeaf) become leaves
};

__device__ __forceinline__ int f2ord(float f) { int i = __float_as_int(f); return i >= 0 ? i : i ^ 0x7fffffff; }
__device__ __host__ __forceinline__ float ord2f(int i) { int j = i >= 0 ? i : i ^ 0x7fffffff; float f; memcpy(&f, &j, 4); return f; }

__global__ void lb_bounds(DevArrays A)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    float lo[3] = { FLT_MAX, FLT_MAX, FLT_MAX }, hi[3] = { -FLT_MAX, -FLT_MAX, -FLT_MAX }, c[3] = { 0, 0, 0 }, am = 0.0f;
    const bool live = i < A.n;
    if (live)
    {
        const float* p = A.tri9 + 9 * (size_t)i;
        for (int a = 0; a < 3; a++)
        {
            lo[a] = fminf(fminf(p[a], p[3 + a]), p[6 + a]);
            hi[a] = fmaxf(fmaxf(p[a], p[3 + a]), p[6 + a]);
            c[a] = 0.5f * (lo[a] + hi[a]);
            am = fmaxf(am, fmaxf(fabsf(lo[a]), fabsf(hi[a])));
        }
        A.plo[i] = make_float4(lo[0], lo[1], lo[2], 0.0f);
        A.phi[i] = make_float4(hi[0], hi[1], hi[2], 0.0f);
    }
    for (int a = 0; a < 3; a++)
    {
        float mn = live ? c[a] : FLT_MAX, mx = live ? c[a] : -FLT_MAX;
        for (int o = 16; o > 0; o >>= 1) { mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o)); mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o)); }
        if ((threadIdx.x & 31) == 0 && mn <= mx) { atomicMin(&A.scene[a], f2ord(mn)); atomicMax(&A.scene[3 + a], f2ord(mx)); }
    }
    for (int o = 16; o > 0; o >>= 1) am = fmaxf(am, __shfl_xor_sync(0xffffffffu, am, o));
    if ((threadIdx.x & 31) == 0) atomicMax(&A.scene[6], f2ord(am));
    for (int a = 0; a < 3; a++)
    {
        float mn = live ? lo[a] : FLT_MAX, mx = live ? hi[a] : -FLT_MAX;
        for (int o = 16; o > 0; o >>= 1) { mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o)); mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o)); }
        if ((threadIdx.x & 31) == 0 && mn <= mx) { atomicMin(&A.scene[8 + a], f2ord(mn)); atomicMax(&A.scene[11 + a], f2ord(mx)); }
    }
}

__device__ __forceinline__ unsigned long long spread3(unsigned long long x)       // 21 bits -> every third bit
{
    x &= 0x1fffffull;
    x = (x | x << 32) & 0x1f00000000ffffull;
    x = (x | x << 16) & 0x1f0000ff0000ffull;
    x = (x | x << 8) & 0x100f00f00f00f00full;
    x = (x | x << 4) & 0x10c30c30c30c30c3ull;
    x = (x | x << 2) & 0x1249249249249249ull;
    return x;
}

__global__ void lb_morton(DevArrays A)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= A.n) return;
    const float4 lo = A.plo[i], hi = A.phi[i];
    const float c[3] = { 0.5f * (lo.x + hi.x), 0.5f * (lo.y + hi.y), 0.5f * (lo.z + hi.z) };
    if (A.segregate)
    {
        double d2 = 0.0, s2 = 0.0;
        const float ext[3] = { hi.x - lo.x, hi.y - lo.y, hi.z - lo.z };
        for (int a = 0; a < 3; a++)
        {
            const double se = (double)ord2f(A.scene[11 + a]) - (double)ord2f(A.scene[8 + a]);
            d2 += (double)ext[a] * ext[a]; s2 += se * se;
        }
        if (d2 > 0.0625 * s2)          // box diagonal > 1/4 of the scene's
        {
            A.keys[i] = ~0ull;
            A.vals[i] = i;
            atomicAdd(&A.scene[14], 1);
            return;
        }
    }
    unsigned long long code = 0;
    for (int a = 0; a < 3; a++)
    {
        const double mn = ord2f(A.scene[a]), mx = ord2f(A.scene[3 + a]);
        const double ext = mx - mn;
        double u = ext > 0.0 ? ((double)c[a] - mn) / ext : 0.0;
        u = fmin(fmax(u, 0.0), 1.0);
        const unsigned long long q = (unsigned long long)fmin(u * 2097152.0, 2097151.0);
        code |= spread3(q) << a;
    }
    A.keys[i] = code;
    A.vals[i] = i;
}

// common-prefix length of sorted keys i and j, ties broken by position; -1 outside the array
__device__ __forceinline__ int lb_delta(const unsigned long long* k, int n, int i, int j)
{
    if (j < 0 || j >= n) return -1;
    const unsigned long long a = k[i], b = k[j];
    if (a == b) return 64 + __clz(i ^ j);
    return __clzll((long long)(a ^ b));
}

__global__ void lb_tree(DevArrays A)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int n = A.n;
    if (i >= n - 1) return;
    const unsigned long long* k = A.keys;
    const int d = (lb_delta(k, n, i, i + 1) - lb_delta(k, n, i, i - 1)) >= 0 ? 1 : -1;
    const int dmin = lb_delta(k, n, i, i - d);
    int lmax = 2;
    while (lb_delta(k, n, i, i + lmax * d) > dmin) lmax <<= 1;
    int l = 0;
    for (int t = lmax >> 1; t >= 1; t >>= 1)
        if (lb_delta(k, n, i, i + (l + t) * d) > dmin) l += t;
    const int j = i + l * d;
    const int dnode = lb_delta(k, n, i, j);
    int s = 0;
    for (int t = (l + 1) >> 1;; t = (t + 1) >> 1)
    {
        if (lb_delta(k, n, i, i + (s + t) * d) > dnode) s += t;
        if (t <= 1) break;
    }
    const int gamma = i + s * d + min(d, 0);
    const int lo = min(i, j), hi = max(i, j);
    const int L = (lo == gamma) ? (gamma | kLeafBit) : gamma;
    const int R = (hi == gamma + 1) ? ((gamma + 1) | kLeafBit) : gamma + 1;
    A.left[i] = L; A.right[i] = R; A.first[i] = lo; A.last[i] = hi;
    if (L & kLeafBit) A.parent_leaf[gamma] = i; else A.parent_node[gamma] = i;
    if (R & kLeafBit) A.parent_leaf[gamma + 1] = i; else A.parent_node[gamma + 1] = i;
    if (i == 0) A.parent_node[0] = -1;
}

// one thread per sorted triangle walks up; the second arrival at a node fits its box. Also the depth of every leaf.
__global__ void lb_fit(DevArrays A, int* max_depth)
{
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= A.n) return;
    int node = A.parent_leaf[p];
    int depth = 1;
    bool fitting = true;
    while (node >= 0)
    {
        depth++;
        if (fitting)
        {
            __threadfence();
            if (atomicAdd(&A.visits[node], 1u) == 0u) fitting = false;        // first arrival: the sibling subtree is not done yet
            else
            {
                const int L = A.left[node], R = A.right[node];
                // inner children were written by other threads of this launch: read them at L2 (__ldcg), not through this SM's L1
                const float4 llo = (L & kLeafBit) ? A.plo[A.vals[L & ~kLeafBit]] : __ldcg(A.nlo + L), lhi = (L & kLeafBit) ? A.phi[A.vals[L & ~kLeafBit]] : __ldcg(A.nhi + L);
                const float4 rlo = (R & kLeafBit) ? A.plo[A.vals[R & ~kLeafBit]] : __ldcg(A.nlo + R), rhi = (R & kLeafBit) ? A.phi[A.vals[R & ~kLeafBit]] : __ldcg(A.nhi + R);
                A.nlo[node] = make_float4(fminf(llo.x, rlo.x), fminf(llo.y, rlo.y), fminf(llo.z, rlo.z), 0.0f);
                A.nhi[node] = make_float4(fmaxf(lhi.x, rhi.x), fmaxf(lhi.y, rhi.y), fmaxf(lhi.z, rhi.z), 0.0f);
            }
        }
        node = A.parent_node[node];
    }
    for (int o = 16; o > 0; o >>= 1) depth = max(depth, __shfl_xor_sync(0xffffffffu, depth, o));
    if ((threadIdx.x & 31) == 0) atomicMax(max_depth, depth);
}

// ---- parallel locally-ordered clustering -----------------------------------------------------------------------------------------
constexpr int kPlocRadius = 32;          // largest search radius (shared-memory halo); the radius in use is a launch argument
constexpr int kPlocSearchRadius = 16;    // the radius in use
constexpr int kPlocBlock = 256;

struct PlocArrays
{
    int *cid[2];                   // cluster -> tree reference (inner node index, or sorted position | kLeafBit), ping-pong
    float4 *clo[2], *chi[2];       // cluster boxes, ping-pong
    int* nn;                       // nearest neighbour (cluster index)
    int* valid;                    // 1: the cluster survives this round (merged clusters live at the lower index)
    int* pos;                      // exclusive scan of valid
    int* size;                     // per inner node: triangles below
    int* next_node;                // next free inner node index (counts down to 0: the root is created last)
};

__device__ __forceinline__ float union_area(float4 alo, float4 ahi, float4 blo, float4 bhi)
{
    const float dx = fmaxf(ahi.x, bhi.x) - fminf(alo.x, blo.x), dy = fmaxf(ahi.y, bhi.y) - fminf(alo.y, blo.y), dz = fmaxf(ahi.z, bhi.z) - fminf(alo.z, blo.z);
    return dx * dy + dy * dz + dz * dx;
}

// nearest neighbour within kPlocRadius places. Pairs are ordered by (area, distance along the curve, parity of the lower index,
// lower index): a total order, so the globally best pair is always mutual and every round merges at least one pair; the
// parity term makes runs of identical boxes (duplicated geometry) pair up as (0,1) (2,3) ... instead of one pair per round.
__device__ __forceinline__ bool pl_pair_less(float a, int i, int j, float b, int k)
{
    if (a != b) return a < b;
    const int dj = abs(i - j), dk = abs(i - k);
    if (dj != dk) return dj < dk;
    const int mj = min(i, j), mk = min(i, k);
    if ((mj & 1) != (mk & 1)) return (mj & 1) == 0;
    return mj < mk;
}

__global__ void __launch_bounds__(kPlocBlock) pl_nearest(const float4* __restrict__ clo, const float4* __restrict__ chi, int n, int radius, int* __restrict__ nn)
{
    __shared__ float4 slo[kPlocBlock + 2 * kPlocRadius], shi[kPlocBlock + 2 * kPlocRadius];
    const int base = blockIdx.x * kPlocBlock - kPlocRadius;
    for (int t = threadIdx.x; t < kPlocBlock + 2 * kPlocRadius; t += kPlocBlock)
    {
        const int g = base + t;
        if (g >= 0 && g < n) { slo[t] = clo[g]; shi[t] = chi[g]; }
    }
    __syncthreads();
    const int i = blockIdx.x * kPlocBlock + threadIdx.x;
    if (i >= n) return;
    const float4 lo = slo[threadIdx.x + kPlocRadius], hi = shi[threadIdx.x + kPlocRadius];
    float best = FLT_MAX; int bj = -1;
    for (int d = -radius; d <= radius; d++)
    {
        const int j = i + d;
        if (d == 0 || j < 0 || j >= n) continue;
        float a = union_area(lo, hi, slo[threadIdx.x + kPlocRadius + d], shi[threadIdx.x + kPlocRadius + d]);
        if (!(a == a)) a = FLT_MAX;                                   // NaN boxes (non-finite input) sort last
        if (bj < 0 || pl_pair_less(a, i, j, best, bj)) { best = a; bj = j; }
    }
    nn[i] = bj;
}

__global__ void pl_merge(DevArrays A, PlocArrays P, int cur, int n)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int j = P.nn[i];
    if (j < 0 || P.nn[j] != i) { P.valid[i] = 1; return; }          // no mutual neighbour this round: carried over unchanged
    if (i > j) { P.valid[i] = 0; return; }                         // the pair lives on at the lower index
    const int node = atomicSub(P.next_node, 1);
    const int L = P.cid[cur][i], R = P.cid[cur][j];
    A.left[node] = L; A.right[node] = R;
    if (L & kLeafBit) A.parent_leaf[L & ~kLeafBit] = node; else A.parent_node[L] = node;
    if (R & kLeafBit) A.parent_leaf[R & ~kLeafBit] = node; else A.parent_node[R] = node;
    const float4 alo = P.clo[cur][i], ahi = P.chi[cur][i], blo = P.clo[cur][j], bhi = P.chi[cur][j];
    const float4 lo = make_float4(fminf(alo.x, blo.x), fminf(alo.y, blo.y), fminf(alo.z, blo.z), 0.0f);
    const float4 hi = make_float4(fmaxf(ahi.x, bhi.x), fmaxf(ahi.y, bhi.y), fmaxf(ahi.z, bhi.z), 0.0f);
    A.nlo[node] = lo; A.nhi[node] = hi;
    P.size[node] = ((L & kLeafBit) ? 1 : P.size[L]) + ((R & kLeafBit) ? 1 : P.size[R]);
    P.cid[cur][i] = node; P.clo[cur][i] = lo; P.chi[cur][i] = hi;
    P.valid[i] = 1;
}

__global__ void pl_compact(PlocArrays P, int cur, int n)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || !P.valid[i]) return;
    const int o = P.pos[i];
    P.cid[cur ^ 1][o] = P.cid[cur][i]; P.clo[cur ^ 1][o] = P.clo[cur][i]; P.chi[cur ^ 1][o] = P.chi[cur][i];
}

// triangles below every remaining cluster (for the host's top-level sweep)
__global__ void pl_cluster_sizes(const int* cid, const int* size, int nc, int* out)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < nc) out[i] = (cid[i] & kLeafBit) ? 1 : size[cid[i]];
}

__global__ void pl_init(DevArrays A, PlocArrays P)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= A.n) return;
    const int t = A.vals[i];
    P.cid[0][i] = i | kLeafBit; P.clo[0][i] = A.plo[t]; P.chi[0][i] = A.phi[t];
}

// depth-first layout, one tree level per launch: a node's triangles occupy [first, first + size) of the final order, its left
// subtree first; pre[] = the node's rank in a depth-first pre-order of the inner nodes (root 0, left child next, right child after
// the left subtree). frontier: inner nodes of this level; leaves get their final position in newpos.
__global__ void pl_layout(DevArrays A, PlocArrays P, const int* frontier, int n_front, int* next_frontier, int* n_next, int* newpos, int* pre)
{
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n_front) return;
    const int node = frontier[k];
    const int first = A.first[node];
    A.last[node] = first + P.size[node] - 1;
    const int L = A.left[node], R = A.right[node];
    const int ls = (L & kLeafBit) ? 1 : P.size[L];
    if (L & kLeafBit) newpos[L & ~kLeafBit] = first; else { A.first[L] = first; pre[L] = pre[node] + 1; next_frontier[atomicAdd(n_next, 1)] = L; }
    if (R & kLeafBit) newpos[R & ~kLeafBit] = first + ls; else { A.first[R] = first + ls; pre[R] = pre[node] + ls; next_frontier[atomicAdd(n_next, 1)] = R; }
}

// leaves move to their depth-first positions: the triangle order (vals) is permuted
__global__ void pl_permute_vals(const int* vals, const int* newpos, int n, int* vals_out)
{
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p < n) vals_out[newpos[p]] = vals[p];
}

// inner nodes move to their pre-order ranks (clustering numbered them in merge order, i.e. scattered in memory: every step of a
// traversal would be a cache miss — the binary layout's records are emitted in node order) and their references follow
__global__ void pl_relabel_nodes(DevArrays A, const int* pre, const int* newpos, int* o_left, int* o_right, int* o_first, int* o_last,
                                 float4* o_lo, float4* o_hi)
{
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= A.n - 1) return;
    const int nv = pre[v];
    const int L = A.left[v], R = A.right[v];
    o_left[nv] = (L & kLeafBit) ? (newpos[L & ~kLeafBit] | kLeafBit) : pre[L];
    o_right[nv] = (R & kLeafBit) ? (newpos[R & ~kLeafBit] | kLeafBit) : pre[R];
    o_first[nv] = A.first[v]; o_last[nv] = A.last[v];
    o_lo[nv] = A.nlo[v]; o_hi[nv] = A.nhi[v];
}

// ---- 8-ary collapse ------------------------------------------------------------------------------------------------------------
struct WideArrays
{
    int* root;            // wide node -> radix-tree node it was opened from
    int* slots;           // [8 per wide node] child reference by octant slot, kEmpty when unused
    int* n_inner;         // inner children per wide node
    int* n_tris;          // triangles in leaf children per wide node
    int* child_base;
    int* tri_base;
    int* node_first;      // radix-tree node collapsed into a leaf -> first slot of its triangles in the final stream
    int* leaf_first;      // sorted triangle position that is a leaf child on its own -> its slot in the final stream
};
constexpr int kEmpty = -1;

__device__ __forceinline__ int ref_size(const DevArrays& A, int ref) { return (ref & kLeafBit) ? 1 : A.last[ref] - A.first[ref] + 1; }
__device__ __forceinline__ bool ref_inner(const DevArrays& A, int ref) { return ref_size(A, ref) > A.leaf_max; }
__device__ __forceinline__ void ref_box(const DevArrays& A, int ref, float4& lo, float4& hi)
{
    if (ref & kLeafBit) { const int t = A.vals[ref & ~kLeafBit]; lo = A.plo[t]; hi = A.phi[t]; }
    else { lo = A.nlo[ref]; hi = A.nhi[ref]; }
}
__device__ __forceinline__ float half_area(float4 lo, float4 hi)
{
    const float dx = hi.x - lo.x, dy = hi.y - lo.y, dz = hi.z - lo.z;
    return dx * dy + dy * dz + dz * dx;
}

// wide nodes [begin, end): open the largest inner child until 8, give every child its octant slot
__global__ void lw_expand(DevArrays A, WideArrays W, int begin, int end)
{
    const int w = begin + blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= end) return;
    const int rn = W.root[w];
    int kids[8]; int nk = 0;
    kids[nk++] = A.left[rn]; kids[nk++] = A.right[rn];
    while (nk < 8)
    {
        int best = -1; float best_area = -1.0f;
        for (int k = 0; k < nk; k++)
        {
            if (!ref_inner(A, kids[k])) continue;
            float4 lo, hi; ref_box(A, kids[k], lo, hi);
            const float ar = half_area(lo, hi);
            if (ar > best_area) { best_area = ar; best = k; }
        }
        if (best < 0) break;
        const int c = kids[best];
        kids[best] = A.left[c]; kids[nk++] = A.right[c];
    }
    const float4 blo = A.nlo[rn], bhi = A.nhi[rn];
    const float nc[3] = { 0.5f * (blo.x + bhi.x), 0.5f * (blo.y + bhi.y), 0.5f * (blo.z + bhi.z) };
    float cost[8][8];
    for (int k = 0; k < nk; k++)
    {
        float4 lo, hi; ref_box(A, kids[k], lo, hi);
        const float cc[3] = { 0.5f * (lo.x + hi.x) - nc[0], 0.5f * (lo.y + hi.y) - nc[1], 0.5f * (lo.z + hi.z) - nc[2] };
        for (int s = 0; s < 8; s++) cost[k][s] = ((s & 1) ? cc[0] : -cc[0]) + ((s & 2) ? cc[1] : -cc[1]) + ((s & 4) ? cc[2] : -cc[2]);
    }
    int slot_ref[8];
    for (int s = 0; s < 8; s++) slot_ref[s] = kEmpty;
    unsigned int kid_done = 0, slot_used = 0;
    for (int round = 0; round < nk; round++)
    {
        int bk = -1, bs = -1; float bc = -FLT_MAX;
        for (int k = 0; k < nk; k++)
        {
            if (kid_done & (1u << k)) continue;
            for (int s = 0; s < 8; s++)
                if (!(slot_used & (1u << s)) && (bk < 0 || cost[k][s] > bc)) { bc = cost[k][s]; bk = k; bs = s; }
        }
        slot_ref[bs] = kids[bk]; kid_done |= 1u << bk; slot_used |= 1u << bs;
    }
    int ni = 0, nt = 0;
    for (int s = 0; s < 8; s++)
    {
        W.slots[8 * (size_t)w + s] = slot_ref[s];
        if (slot_ref[s] == kEmpty) continue;
        if (ref_inner(A, slot_ref[s])) ni++; else nt += ref_size(A, slot_ref[s]);
    }
    W.n_inner[w] = ni; W.n_tris[w] = nt;
}

__global__ void lw_shift(int* p, int n, int by)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] += by;
}

// the inner children of wide nodes [begin, end) become the wide nodes of the next level (child_base already scanned)
__global__ void lw_link(DevArrays A, WideArrays W, int begin, int end)
{
    const int w = begin + blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= end) return;
    int at = W.child_base[w];
    for (int s = 0; s < 8; s++)
    {
        const int r = W.slots[8 * (size_t)w + s];
        if (r != kEmpty && ref_inner(A, r)) W.root[at++] = r;
    }
}

// quantised node + its leaf children's triangles (device twin of WideBuilder::quantise_axis / emit in bvh_build.cpp; the frame and the
// quantisation are wide_quantise, which the refit shares)
__global__ void lw_emit(DevArrays A, WideArrays W, int n_wide, float abs_pad, WideNode* nodes, float4* tris, int* overflow)
{
    const int w = blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= n_wide) return;
    WideNode node;
    memset(&node, 0, sizeof(node));
    node.child_base = (uint32_t)W.child_base[w];
    node.tri_base = (uint32_t)W.tri_base[w];
    unsigned used = 0;
    float klo[8][3], khi[8][3];
    int at = W.tri_base[w];
    for (int s = 0; s < 8; s++)
    {
        const int r = W.slots[8 * (size_t)w + s];
        if (r == kEmpty) continue;
        used |= 1u << s;
        float4 lo, hi; ref_box(A, r, lo, hi);
        const float l3[3] = { lo.x, lo.y, lo.z }, h3[3] = { hi.x, hi.y, hi.z };
        for (int a = 0; a < 3; a++)
        {
            const float pad = box_pad_dev(l3[a], h3[a], abs_pad);
            klo[s][a] = l3[a] - pad; khi[s][a] = h3[a] + pad;
        }
        if (ref_inner(A, r)) { node.imask |= (uint8_t)(1u << s); continue; }
        const int cnt = ref_size(A, r);
        const int p0 = (r & kLeafBit) ? (r & ~kLeafBit) : A.first[r];
        if (r & kLeafBit) W.leaf_first[p0] = at; else W.node_first[r] = at;
        for (int i = 0; i < cnt; i++) emit_triangle(A.tri9, A.vals[p0 + i], tris + 3 * (size_t)(at + i));
        node.valid24 |= ((1u << cnt) - 1u) << (3 * s);
        at += cnt;
    }
    wide_quantise(node, klo, khi, used, overflow);
    nodes[w] = node;
}

// the outsized triangles behind the tree's stream records (emit_triangle, as every other record), and their vertices for the host's
// top-level arithmetic
__global__ void lw_emit_extra(const float* tri9, const int* ids, int n, float4* tris, float* extra9)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    emit_triangle(tri9, ids[i], tris + 3 * (size_t)i);
    for (int k = 0; k < 9; k++) extra9[9 * i + k] = tri9[9 * (size_t)ids[i] + k];
}

__global__ void k_slot_of_prim(const float4* tris, int n, int* slot_of_prim)
{
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j < n) slot_of_prim[__float_as_int(tris[3 * (size_t)j].w)] = j;
}

// ---- binary records over the same tree and the same triangle stream ---------------------------------------------------------------------
__global__ void lb_mark_live(DevArrays A, int* live)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < A.n - 1) live[i] = (A.last[i] - A.first[i] + 1) > A.leaf_max ? 1 : 0;
}

__global__ void lb_emit(DevArrays A, WideArrays W, const int* live, const int* axis_idx, float abs_pad, AxisNode* axis)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= A.n - 1 || !live[i]) return;
    AxisNode an;
    for (int side = 0; side < 2; side++)
    {
        const int r = side ? A.right[i] : A.left[i];
        float4 lo, hi; ref_box(A, r, lo, hi);
        float* olo = side ? an.r_lo : an.l_lo; float* ohi = side ? an.r_hi : an.l_hi;
        const float l3[3] = { lo.x, lo.y, lo.z }, h3[3] = { hi.x, hi.y, hi.z };
        for (int a = 0; a < 3; a++)
        {
            const float pad = box_pad_dev(l3[a], h3[a], abs_pad);
            olo[a] = l3[a] - pad; ohi[a] = h3[a] + pad;
        }
        int ref, count = 0;
        if (ref_inner(A, r)) ref = axis_idx[r];
        else
        {
            count = ref_size(A, r);
            const int first = (r & kLeafBit) ? W.leaf_first[r & ~kLeafBit] : W.node_first[r];
            ref = ~((first << 4) | count);
        }
        if (side) { an.r_ref = ref; an.r_count = count; } else { an.l_ref = ref; an.l_count = count; }
    }
    axis[axis_idx[i]] = an;
}

// ---- top of the clustered tree: surface-area-heuristic sweep on the host -----------------------------------------------------------
// Agglomerative clustering builds excellent lower levels and mediocre upper ones (few, large clusters seen through a fixed window
// along the Morton curve), and every ray walks the upper levels. When at most kPlocTop clusters are left the clustering stops and
// the tree above them is built top-down by a full SAH sweep (sort by centroid on every axis, cost = area x triangles below): a few
// thousand boxes, well under a millisecond on the host.
constexpr int kPlocTop = 1024;
struct TopCluster { float lo[3], hi[3]; int ref, size; };

struct TopBuilder
{
    std::vector<TopCluster> c;
    std::vector<int> left, right, size;
    std::vector<float4> nlo, nhi;
    int next = 0;

    static double area(const float* lo, const float* hi)
    {
        const double dx = (double)hi[0] - lo[0], dy = (double)hi[1] - lo[1], dz = (double)hi[2] - lo[2];
        return dx * dy + dy * dz + dz * dx;
    }

    // builds the subtree over c[begin, end) (reordered in place); returns its reference
    int build(int begin, int end)
    {
        if (end - begin == 1) return c[(size_t)begin].ref;
        const int id = next++;
        float lo[3] = { FLT_MAX, FLT_MAX, FLT_MAX }, hi[3] = { -FLT_MAX, -FLT_MAX, -FLT_MAX };
        int total = 0;
        for (int i = begin; i < end; i++)
        {
            for (int a = 0; a < 3; a++) { lo[a] = std::min(lo[a], c[(size_t)i].lo[a]); hi[a] = std::max(hi[a], c[(size_t)i].hi[a]); }
            total += c[(size_t)i].size;
        }
        nlo[(size_t)id] = make_float4(lo[0], lo[1], lo[2], 0.0f); nhi[(size_t)id] = make_float4(hi[0], hi[1], hi[2], 0.0f);
        size[(size_t)id] = total;
        const int n = end - begin;
        int best_axis = -1, best_split = -1;
        double best_cost = DBL_MAX;
        std::vector<double> right_area((size_t)n);
        std::vector<int> right_cnt((size_t)n);
        for (int axis = 0; axis < 3; axis++)
        {
            std::sort(c.begin() + begin, c.begin() + end, [axis](const TopCluster& p, const TopCluster& q) { return p.lo[axis] + p.hi[axis] < q.lo[axis] + q.hi[axis]; });
            float rlo[3] = { FLT_MAX, FLT_MAX, FLT_MAX }, rhi[3] = { -FLT_MAX, -FLT_MAX, -FLT_MAX };
            int rc = 0;
            for (int i = n - 1; i >= 1; i--)
            {
                const TopCluster& t = c[(size_t)(begin + i)];
                for (int a = 0; a < 3; a++) { rlo[a] = std::min(rlo[a], t.lo[a]); rhi[a] = std::max(rhi[a], t.hi[a]); }
                rc += t.size;
                right_area[(size_t)i] = area(rlo, rhi); right_cnt[(size_t)i] = rc;
            }
            float llo[3] = { FLT_MAX, FLT_MAX, FLT_MAX }, lhi[3] = { -FLT_MAX, -FLT_MAX, -FLT_MAX };
            int lc = 0;
            for (int i = 1; i < n; i++)
            {
                const TopCluster& t = c[(size_t)(begin + i - 1)];
                for (int a = 0; a < 3; a++) { llo[a] = std::min(llo[a], t.lo[a]); lhi[a] = std::max(lhi[a], t.hi[a]); }
                lc += t.size;
                const double cost = area(llo, lhi) * lc + right_area[(size_t)i] * right_cnt[(size_t)i];
                if (cost < best_cost) { best_cost = cost; best_axis = axis; best_split = i; }
            }
        }
        if (best_axis != 2)
            std::sort(c.begin() + begin, c.begin() + end, [best_axis](const TopCluster& p, const TopCluster& q) { return p.lo[best_axis] + p.hi[best_axis] < q.lo[best_axis] + q.hi[best_axis]; });
        const int l = build(begin, begin + best_split), r = build(begin + best_split, end);
        left[(size_t)id] = l; right[(size_t)id] = r;
        return id;
    }
};

struct Pool       // frees everything it handed out
{
    std::vector<void*> p;
    ~Pool() { release(); }
    void release() { for (void* q : p) cudaFree(q); p.clear(); }
    template <typename T> cudaError_t get(T** out, size_t n)
    {
        void* d = nullptr;
        cudaError_t e = cudaMalloc(&d, std::max<size_t>(n, 1) * sizeof(T));
        if (e == cudaSuccess) { p.push_back(d); *out = (T*)d; }
        return e;
    }
};

} // namespace

#define GCU(expr)                                                                                    \
    do {                                                                                             \
        cudaError_t e__ = (expr);                                                                    \
        if (e__ != cudaSuccess) { err = std::string(#expr) + ": " + cudaGetErrorString(e__); return 1; } \
    } while (0)

// 0 = ok; 1 = CUDA error; 2 = the input is outside what this builder handles
static int build_bvh_device_impl(const float* d_tri9, int n_tri, cudaStream_t st, bool use_lbvh, const DeviceTreeAlloc& alloc,
                                 b200rt_bvh_info& info, DeviceBuildCounts& C, std::string& err)
{
    if (n_tri <= kWideMaxLeaf) { err = "fewer than 4 triangles"; return 2; }
    // host <-> device: every copy is counted; a download returns once the host holds it
    auto h2d = [&](void* dst, const void* src, size_t bytes) { C.h2d_bytes += bytes; return cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, st); };
    auto d2h = [&](void* dst, const void* src, size_t bytes) {
        C.d2h_bytes += bytes;
        const cudaError_t e = cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, st);
        return e != cudaSuccess ? e : cudaStreamSynchronize(st);
    };
    Pool pool;
    DevArrays A;
    memset(&A, 0, sizeof(A));
    A.n = n_tri;
    A.leaf_max = kWideMaxLeaf;
    const size_t n = (size_t)n_tri;
    A.tri9 = d_tri9;
    GCU(pool.get(&A.plo, n)); GCU(pool.get(&A.phi, n));
    GCU(pool.get(&A.keys, n)); GCU(pool.get(&A.keys_alt, n)); GCU(pool.get(&A.vals, n)); GCU(pool.get(&A.vals_alt, n));
    GCU(pool.get(&A.left, n)); GCU(pool.get(&A.right, n)); GCU(pool.get(&A.first, n)); GCU(pool.get(&A.last, n));
    GCU(pool.get(&A.parent_node, n)); GCU(pool.get(&A.parent_leaf, n));
    GCU(pool.get(&A.nlo, n)); GCU(pool.get(&A.nhi, n)); GCU(pool.get(&A.visits, n));
    GCU(pool.get(&A.scene, 16));
    int* d_misc = nullptr;                   // [0] max depth, [1] overflow flag
    GCU(pool.get(&d_misc, 4));
    GCU(cudaMemsetAsync(d_misc, 0, 4 * sizeof(int), st));
    GCU(cudaMemsetAsync(A.visits, 0, n * sizeof(unsigned int), st));
    {
        const int init[16] = { INT32_MAX, INT32_MAX, INT32_MAX, INT32_MIN, INT32_MIN, INT32_MIN, INT32_MIN, 0,
                               INT32_MAX, INT32_MAX, INT32_MAX, INT32_MIN, INT32_MIN, INT32_MIN, 0, 0 };
        GCU(h2d(A.scene, init, sizeof(init)));
    }
    const int tb = 256;
    int grid_n = (n_tri + tb - 1) / tb;
    lb_bounds<<<grid_n, tb, 0, st>>>(A); C.launches++;
    size_t sort_bytes = 0;
    {
        cub::DoubleBuffer<unsigned long long> dk(A.keys, A.keys_alt);
        cub::DoubleBuffer<int> dv(A.vals, A.vals_alt);
        GCU(cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, dk, dv, n_tri, 0, 64, st));
    }
    char* sort_tmp = nullptr;
    GCU(pool.get(&sort_tmp, sort_bytes));
    int n_large = 0;
    for (int attempt = 0; attempt < 2; attempt++)
    {
        // first with the outsized triangles given the largest key (they sort to the end and stay out of the tree); if there are
        // too many of them for a few top-level nodes, or too few others for a tree, once more with everything in the tree
        A.segregate = attempt == 0 ? 1 : 0;
        lb_morton<<<grid_n, tb, 0, st>>>(A); C.launches++;
        cub::DoubleBuffer<unsigned long long> dk(A.keys, A.keys_alt);
        cub::DoubleBuffer<int> dv(A.vals, A.vals_alt);
        GCU(cub::DeviceRadixSort::SortPairs(sort_tmp, sort_bytes, dk, dv, n_tri, 0, 64, st)); C.launches++;
        A.keys = dk.Current(); A.keys_alt = dk.Alternate(); A.vals = dv.Current(); A.vals_alt = dv.Alternate();
        n_large = 0;
        if (attempt == 0) GCU(d2h(&n_large, A.scene + 14, sizeof(int)));
        if (n_large <= 45 && n_tri - n_large > kWideMaxLeaf) break;
    }
    std::vector<int> large_ids((size_t)n_large);
    if (n_large) GCU(d2h(large_ids.data(), A.vals + (n_tri - n_large), (size_t)n_large * sizeof(int)));
    const int n_all = n_tri;
    n_tri -= n_large;                         // the tree is built over the first n_tri sorted triangles
    A.n = n_tri;
    grid_n = (n_tri + tb - 1) / tb;
    if (use_lbvh)
    {
        lb_tree<<<grid_n, tb, 0, st>>>(A);
        lb_fit<<<grid_n, tb, 0, st>>>(A, d_misc);
        C.launches += 2;
    }
    else
    {
        PlocArrays P;
        memset(&P, 0, sizeof(P));
        for (int b = 0; b < 2; b++) { GCU(pool.get(&P.cid[b], n)); GCU(pool.get(&P.clo[b], n)); GCU(pool.get(&P.chi[b], n)); }
        GCU(pool.get(&P.nn, n)); GCU(pool.get(&P.valid, n)); GCU(pool.get(&P.pos, n)); GCU(pool.get(&P.size, n)); GCU(pool.get(&P.next_node, 1));
        size_t pscan_bytes = 0;
        GCU(cub::DeviceScan::ExclusiveSum(nullptr, pscan_bytes, P.valid, P.pos, n_tri, st));
        char* pscan_tmp = nullptr;
        GCU(pool.get(&pscan_tmp, pscan_bytes));
        const int first_node = n_tri - 2;
        GCU(h2d(P.next_node, &first_node, sizeof(int)));
        pl_init<<<grid_n, tb, 0, st>>>(A, P); C.launches++;
        int nc = n_tri, cur = 0, rounds = 0;
        while (nc > kPlocTop)
        {
            if (++rounds > 512) { err = "clustering needs more than 512 rounds (a size gradient along the Morton curve merges one pair per round)"; return 2; }
            const int g = (nc + kPlocBlock - 1) / kPlocBlock;
            pl_nearest<<<g, kPlocBlock, 0, st>>>(P.clo[cur], P.chi[cur], nc, kPlocSearchRadius, P.nn);
            pl_merge<<<g, kPlocBlock, 0, st>>>(A, P, cur, nc);
            GCU(cub::DeviceScan::ExclusiveSum(pscan_tmp, pscan_bytes, P.valid, P.pos, nc, st));
            pl_compact<<<g, kPlocBlock, 0, st>>>(P, cur, nc);
            C.launches += 4;
            int last[2] = { 0, 0 };
            GCU(d2h(&last[0], P.pos + nc - 1, sizeof(int)));
            GCU(d2h(&last[1], P.valid + nc - 1, sizeof(int)));
            const int next = last[0] + last[1];
            if (next >= nc) { err = "clustering round merged nothing"; return 1; }
            nc = next; cur ^= 1;
        }
        if (nc > 1)
        {
            // the tree above the remaining clusters: SAH sweep on the host, into the node indices clustering has not used (0 .. nc - 2)
            std::vector<int> h_cid((size_t)nc);
            std::vector<float4> h_lo((size_t)nc), h_hi((size_t)nc);
            std::vector<int> h_size((size_t)nc);
            pl_cluster_sizes<<<(nc + 255) / 256, 256, 0, st>>>(P.cid[cur], P.size, nc, P.nn); C.launches++;
            GCU(d2h(h_size.data(), P.nn, (size_t)nc * sizeof(int)));
            GCU(d2h(h_cid.data(), P.cid[cur], (size_t)nc * sizeof(int)));
            GCU(d2h(h_lo.data(), P.clo[cur], (size_t)nc * sizeof(float4)));
            GCU(d2h(h_hi.data(), P.chi[cur], (size_t)nc * sizeof(float4)));
            TopBuilder T;
            T.c.resize((size_t)nc);
            for (int i = 0; i < nc; i++)
            {
                TopCluster& t = T.c[(size_t)i];
                t.lo[0] = h_lo[(size_t)i].x; t.lo[1] = h_lo[(size_t)i].y; t.lo[2] = h_lo[(size_t)i].z;
                t.hi[0] = h_hi[(size_t)i].x; t.hi[1] = h_hi[(size_t)i].y; t.hi[2] = h_hi[(size_t)i].z;
                t.ref = h_cid[(size_t)i];
                t.size = h_size[(size_t)i];
            }
            const size_t nt = (size_t)nc - 1;
            T.left.resize(nt); T.right.resize(nt); T.size.resize(nt); T.nlo.resize(nt); T.nhi.resize(nt);
            const int root = T.build(0, nc);
            if (root != 0 || T.next != nc - 1) { err = "top-level build produced an inconsistent tree"; return 1; }
            GCU(h2d(A.left, T.left.data(), nt * sizeof(int)));
            GCU(h2d(A.right, T.right.data(), nt * sizeof(int)));
            GCU(h2d(P.size, T.size.data(), nt * sizeof(int)));
            GCU(h2d(A.nlo, T.nlo.data(), nt * sizeof(float4)));
            GCU(h2d(A.nhi, T.nhi.data(), nt * sizeof(float4)));
            GCU(cudaStreamSynchronize(st));          // T's vectors are the sources of the copies above
        }
        // the root is the node created last: index 0
        {
            const int none = -1, zero = 0;
            GCU(h2d(A.parent_node, &none, sizeof(int)));
            GCU(h2d(A.first, &zero, sizeof(int)));
        }
        // depth-first layout level by level (the clustering arrays are free again: frontiers, the leaf permutation, the relabelled nodes)
        int* front[2] = { P.cid[0], P.cid[1] };
        int* d_nnext = P.next_node;
        int* newpos = P.nn;
        int* pre = reinterpret_cast<int*>(A.visits);
        {
            const int zero = 0;
            GCU(h2d(front[0], &zero, sizeof(int)));
            GCU(h2d(pre, &zero, sizeof(int)));
        }
        int n_front = 1, f = 0, depth = 1;
        while (n_front > 0)
        {
            depth++;
            if (depth > 4096) { err = "layout did not terminate"; return 1; }
            GCU(cudaMemsetAsync(d_nnext, 0, sizeof(int), st));
            pl_layout<<<(n_front + 255) / 256, 256, 0, st>>>(A, P, front[f], n_front, front[f ^ 1], d_nnext, newpos, pre); C.launches++;
            GCU(d2h(&n_front, d_nnext, sizeof(int)));
            f ^= 1;
        }
        GCU(h2d(d_misc, &depth, sizeof(int)));
        pl_permute_vals<<<grid_n, tb, 0, st>>>(A.vals, newpos, n_tri, A.vals_alt); C.launches++;
        // the outsized triangles behind the tree keep their places in the order
        if (n_large) GCU(cudaMemcpyAsync(A.vals_alt + n_tri, A.vals + n_tri, (size_t)n_large * sizeof(int), cudaMemcpyDeviceToDevice, st));
        pl_relabel_nodes<<<grid_n, tb, 0, st>>>(A, pre, newpos, A.parent_node, A.parent_leaf, P.pos, P.valid, P.clo[0], P.chi[0]); C.launches++;
        std::swap(A.vals, A.vals_alt);
        A.left = A.parent_node; A.right = A.parent_leaf; A.first = P.pos; A.last = P.valid; A.nlo = P.clo[0]; A.nhi = P.chi[0];
    }
    int scene_h[8];
    int misc_h[4];
    GCU(d2h(scene_h, A.scene, sizeof(scene_h)));
    GCU(d2h(misc_h, d_misc, sizeof(misc_h)));
    if (misc_h[0] > kMaxTraversalDepth) { err = "radix tree deeper than the traversal stack (" + std::to_string(misc_h[0]) + ")"; return 2; }
    float scene_abs = ord2f(scene_h[6]);
    if (!(scene_abs < FLT_MAX)) scene_abs = 1.0f;
    const float abs_pad = 2e-6f * scene_abs + 1e-30f;

    // 8-ary collapse, one level at a time
    WideArrays W;
    memset(&W, 0, sizeof(W));
    // wide nodes are radix-tree inner nodes: fewer than n
    GCU(pool.get(&W.root, n)); GCU(pool.get(&W.slots, 8 * n)); GCU(pool.get(&W.n_inner, n)); GCU(pool.get(&W.n_tris, n));
    GCU(pool.get(&W.child_base, n)); GCU(pool.get(&W.tri_base, n)); GCU(pool.get(&W.node_first, n)); GCU(pool.get(&W.leaf_first, n));
    size_t scan_bytes = 0;
    GCU(cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, W.n_inner, W.child_base, n_tri, st));
    char* scan_tmp = nullptr;
    GCU(pool.get(&scan_tmp, scan_bytes));
    {
        const int zero = 0;
        GCU(h2d(W.root, &zero, sizeof(int)));
    }
    int begin = 0, end = 1, wide_depth = 0;
    while (begin < end)
    {
        wide_depth++;
        const int cnt = end - begin, g = (cnt + 127) / 128;
        lw_expand<<<g, 128, 0, st>>>(A, W, begin, end);
        GCU(cub::DeviceScan::ExclusiveSum(scan_tmp, scan_bytes, W.n_inner + begin, W.child_base + begin, cnt, st));
        C.launches += 2;
        int last[2] = { 0, 0 };
        GCU(d2h(&last[0], W.child_base + end - 1, sizeof(int)));
        GCU(d2h(&last[1], W.n_inner + end - 1, sizeof(int)));
        const int next_cnt = last[0] + last[1];
        if (wide_depth > kMaxTraversalDepth) { err = "wide tree deeper than the traversal stack"; return 2; }
        if ((size_t)end + next_cnt > n) { err = "wide node count exceeds its bound"; return 1; }
        lw_shift<<<g, 128, 0, st>>>(W.child_base + begin, cnt, end);      // the scan is relative to the level's first child, which gets index `end`
        lw_link<<<g, 128, 0, st>>>(A, W, begin, end);
        C.launches += 2;
        begin = end; end += next_cnt;
    }
    const int n_wide = end;
    GCU(cub::DeviceScan::ExclusiveSum(scan_tmp, scan_bytes, W.n_tris, W.tri_base, n_wide, st));

    // binary records: which radix-tree nodes stay inner records, and their record indices
    int *d_live = nullptr, *d_axis_idx = nullptr;
    GCU(pool.get(&d_live, n)); GCU(pool.get(&d_axis_idx, n));
    lb_mark_live<<<grid_n, tb, 0, st>>>(A, d_live);
    GCU(cub::DeviceScan::ExclusiveSum(scan_tmp, scan_bytes, d_live, d_axis_idx, n_tri - 1, st));
    C.launches += 3;
    int last_axis[2] = { 0, 0 };
    GCU(d2h(&last_axis[0], d_axis_idx + (n_tri - 2), sizeof(int)));
    GCU(d2h(&last_axis[1], d_live + (n_tri - 2), sizeof(int)));
    const int n_axis = last_axis[0] + last_axis[1];

    // the caller's arrays, with room for the top level over the outsized triangles
    const int n_top_wide = n_large ? top_level_wide(n_large) : 0, n_top_axis = n_large ? top_level_axis(n_large) : 0;
    DeviceTree out;
    GCU(alloc((size_t)n_wide + n_top_wide, (size_t)n_axis + n_top_axis, out));
    WideNode* d_wide = reinterpret_cast<WideNode*>(out.wide_and_tris);
    float4* d_tris = out.wide_and_tris + 5 * ((size_t)n_wide + n_top_wide);
    lw_emit<<<(n_wide + 127) / 128, 128, 0, st>>>(A, W, n_wide, abs_pad, d_wide, d_tris, d_misc + 1);
    lb_emit<<<grid_n, tb, 0, st>>>(A, W, d_live, d_axis_idx, abs_pad, out.axis);
    C.launches += 2;
    GCU(d2h(misc_h, d_misc, sizeof(misc_h)));
    GCU(cudaGetLastError());
    if (misc_h[1]) { err = "wide BVH quantisation overflow"; return 1; }

    memset(&info, 0, sizeof(info));
    info.n_triangles = n_all;
    info.n_inner_nodes = n_axis;
    info.n_leaves = n_axis + 1;
    info.max_leaf_size = kWideMaxLeaf;
    info.max_depth = misc_h[0];
    info.has_diag_slabs = 0;
    info.sah_cost = 0.0;
    info.n_wide_nodes = n_wide;
    info.wide_max_depth = wide_depth;
    if (n_large)
    {
        // the outsized triangles' stream records on the device; record 0 of both layouts and their vertices to the host, which works
        // out the few top-level records; those records back
        std::sort(large_ids.begin(), large_ids.end());
        int* d_ids = nullptr; float* d_extra9 = nullptr;
        GCU(pool.get(&d_ids, (size_t)n_large)); GCU(pool.get(&d_extra9, 9 * (size_t)n_large));
        GCU(h2d(d_ids, large_ids.data(), (size_t)n_large * sizeof(int)));
        lw_emit_extra<<<1, 64, 0, st>>>(d_tri9, d_ids, n_large, d_tris + 3 * (size_t)n_tri, d_extra9); C.launches++;
        std::vector<float> extra9(9 * (size_t)n_large);
        WideNode w0; AxisNode a0;
        GCU(d2h(extra9.data(), d_extra9, extra9.size() * sizeof(float)));
        GCU(d2h(&w0, d_wide, sizeof(w0)));
        GCU(d2h(&a0, out.axis, sizeof(a0)));
        TopLevel top;
        try { make_top_level(w0, a0, (size_t)n_wide, (size_t)n_axis, (size_t)n_tri, extra9.data(), n_large, abs_pad, top, info); }
        catch (const std::exception& e) { err = e.what(); return 1; }
        GCU(h2d(d_wide, top.wide.data(), sizeof(WideNode)));
        GCU(h2d(d_wide + n_wide, top.wide.data() + 1, (top.wide.size() - 1) * sizeof(WideNode)));
        GCU(h2d(out.axis, top.axis.data(), sizeof(AxisNode)));
        GCU(h2d(out.axis + n_axis, top.axis.data() + 1, (top.axis.size() - 1) * sizeof(AxisNode)));
        GCU(cudaStreamSynchronize(st));              // top's vectors are the sources of the copies above
        if (info.max_depth > kMaxTraversalDepth || info.wide_max_depth > kMaxTraversalDepth) { err = "tree deeper than the traversal stack"; return 2; }
    }
    GCU(cudaStreamSynchronize(st));
    return 0;
}

int build_bvh_device(const float* d_tri9, int n_tri, cudaStream_t st, const DeviceTreeAlloc& alloc, b200rt_bvh_info& info,
                     DeviceBuildCounts& counts, std::string& err)
{
    int rc = build_bvh_device_impl(d_tri9, n_tri, st, false, alloc, info, counts, err);
    if (rc == 2) rc = build_bvh_device_impl(d_tri9, n_tri, st, true, alloc, info, counts, err);
    return rc;
}

// 0 = ok; 1 = CUDA error; 2 = the input is outside what this builder handles (caller falls back to the host builder).
int build_flat_bvh_device(const float* tri9_host, int n_tri, int device, FlatBVH& out, std::string& err)
{
    const auto t0 = std::chrono::high_resolution_clock::now();
    if (n_tri <= kWideMaxLeaf) { err = "fewer than 4 triangles"; return 2; }
    GCU(cudaSetDevice(device));
    Pool in;
    float* d_tri9 = nullptr;
    GCU(in.get(&d_tri9, 9 * (size_t)n_tri));
    GCU(cudaMemcpy(d_tri9, tri9_host, 9 * (size_t)n_tri * sizeof(float), cudaMemcpyHostToDevice));
    Pool tree;
    size_t n_wide = 0, n_axis = 0;
    DeviceTree dt;
    const DeviceTreeAlloc alloc = [&](size_t nw, size_t na, DeviceTree& o) {
        tree.release();
        n_wide = nw; n_axis = na;
        cudaError_t e = tree.get(&o.wide_and_tris, 5 * nw + 3 * (size_t)n_tri);
        if (e == cudaSuccess) e = tree.get(&o.axis, na);
        dt = o;
        return e;
    };
    DeviceBuildCounts counts;
    b200rt_bvh_info info;
    const int rc = build_bvh_device(d_tri9, n_tri, 0, alloc, info, counts, err);
    if (rc) return rc;
    out.wide.resize(n_wide); out.tris.resize((size_t)n_tri); out.axis.resize(n_axis); out.diag.clear();
    GCU(cudaMemcpy(out.wide.data(), dt.wide_and_tris, n_wide * sizeof(WideNode), cudaMemcpyDeviceToHost));
    GCU(cudaMemcpy(out.tris.data(), dt.wide_and_tris + 5 * n_wide, (size_t)n_tri * sizeof(LeafTriangle), cudaMemcpyDeviceToHost));
    GCU(cudaMemcpy(out.axis.data(), dt.axis, n_axis * sizeof(AxisNode), cudaMemcpyDeviceToHost));
    out.info = info;
    out.info.build_seconds = std::chrono::duration<double>(std::chrono::high_resolution_clock::now() - t0).count();
    return 0;
}

cudaError_t launch_slot_of_prim(const float4* tris, int n_tri, int* slot_of_prim, cudaStream_t st)
{
    if (n_tri > 0) k_slot_of_prim<<<(n_tri + 255) / 256, 256, 0, st>>>(tris, n_tri, slot_of_prim);
    return cudaGetLastError();
}

} // namespace b200rt
