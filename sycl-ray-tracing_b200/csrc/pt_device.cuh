// Device-side restatement of the reference's per-pixel path (render_kernel.cpp:56-181, :218-759) for sm_100a.
//
// This translation unit is compiled with -fmad=false: every float expression below is evaluated exactly as written
// (IEEE binary32, round-to-nearest, no contraction), which is what the reference's x86-64 build does and what makes
// the primary-ray closest hit bit-exact. Where a fused multiply-add is wanted for speed (slab tests, which only need
// to be conservative) it is requested explicitly with fmaf().
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "../../include/b200rt.h"
#include "device_types.h"

namespace b200rt {

#ifndef B200RT_PI_D
#define B200RT_PI_D 3.14159265358979323846
#define B200RT_1_PI_D 0.31830988618379067154
#endif
#define B200RT_PI_F 3.14159274101257324219f   /* (float)M_PI */

struct v3 { float x, y, z; };
struct col { float r, g, b; };

__device__ __forceinline__ v3 V(float x, float y, float z) { v3 r; r.x = x; r.y = y; r.z = z; return r; }
__device__ __forceinline__ v3 operator+(v3 a, v3 b) { return V(a.x + b.x, a.y + b.y, a.z + b.z); }
__device__ __forceinline__ v3 operator-(v3 a, v3 b) { return V(a.x - b.x, a.y - b.y, a.z - b.z); }
__device__ __forceinline__ v3 operator-(v3 a) { return V(-a.x, -a.y, -a.z); }
__device__ __forceinline__ v3 operator*(float k, v3 a) { return V(k * a.x, k * a.y, k * a.z); }      // vec.h:141-149
__device__ __forceinline__ float dot(v3 u, v3 v) { return u.x * v.x + u.y * v.y + u.z * v.z; }        // vec.h:186-189
__device__ __forceinline__ v3 cross(v3 u, v3 v)                                                       // vec.h:178-184
{
    return V((u.y * v.z) - (u.z * v.y), (u.z * v.x) - (u.x * v.z), (u.x * v.y) - (u.y * v.x));
}
__device__ __forceinline__ float length(v3 v) { return sqrtf(v.x * v.x + v.y * v.y + v.z * v.z); }
__device__ __forceinline__ v3 normalize(v3 v) { float kk = 1.0f / length(v); return kk * v; }         // vec.h:172-176
// std::max / std::min with libstdc++'s exact comparison order (NaN behaviour included)
__device__ __forceinline__ float smax(float a, float b) { return (a < b) ? b : a; }
__device__ __forceinline__ float smin(float a, float b) { return (b < a) ? b : a; }

__device__ __forceinline__ col CO(float r, float g, float b) { col c; c.r = r; c.g = g; c.b = b; return c; }
__device__ __forceinline__ col operator+(col a, col b) { return CO(a.r + b.r, a.g + b.g, a.b + b.b); }
__device__ __forceinline__ col operator*(col a, col b) { return CO(a.r * b.r, a.g * b.g, a.b * b.b); }
__device__ __forceinline__ col operator*(col c, float k) { return CO(c.r * k, c.g * k, c.b * k); }    // color.h:149-157
__device__ __forceinline__ col operator/(col c, float k) { float kk = 1.0f / k; return c * kk; }      // color.h:169-173
__device__ __forceinline__ bool is_black(col c) { return c.r == 0.0f && c.g == 0.0f && c.b == 0.0f; }

// ---- RNG: include/xorshift.h:10-31 ------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t xs_next(uint32_t& s)
{
    uint32_t x = s;
    x ^= x << 13; x ^= x >> 17; x ^= x << 5;
    s = x;
    return x;
}
__device__ __forceinline__ float xs_float(uint32_t& s)
{
    // u32 / (float)UINT_MAX: the divisor rounds to 2^32, so the division is an exact scaling; cap 1 - 1e-6f (xorshift.h:17)
    return smin(__uint2float_rn(xs_next(s)) * 2.3283064365386962890625e-10f, 1.0f - 1.0e-6f);
}
// seed of pixel (x, y): 31 + x*y*spp in wrapping int arithmetic (render_kernel.cpp:77), then 10 warm-up draws (:81-82)
__device__ __forceinline__ uint32_t pixel_rng(int x, int y, int spp)
{
    uint32_t s = 31u + (uint32_t)x * (uint32_t)y * (uint32_t)spp;
#pragma unroll
    for (int i = 0; i < 10; i++) xs_next(s);
    return s;
}

// ---- camera: render_kernel.cpp:56-73, Transform::operator()(Point) mat.cpp:94-111 --------------------------------------
__device__ __forceinline__ v3 xform_point(const float* m, v3 p)
{
    float xt = m[0] * p.x + m[1] * p.y + m[2] * p.z + m[3];
    float yt = m[4] * p.x + m[5] * p.y + m[6] * p.z + m[7];
    float zt = m[8] * p.x + m[9] * p.y + m[10] * p.z + m[11];
    float wt = m[12] * p.x + m[13] * p.y + m[14] * p.z + m[15];
    if (wt == 1.f) return V(xt, yt, zt);
    float w = 1.f / wt;
    return V(xt * w, yt * w, zt * w);
}
__device__ __forceinline__ void camera_ray(const CameraDev& c, float x, float y, v3& o, v3& d)
{
    float x_ndc = x / (float)c.w * 2.0f - 1.0f;
    x_ndc *= (float)c.w / (float)c.h;
    float y_ndc = y / (float)c.h * 2.0f - 1.0f;
    o = xform_point(c.m, V(0.0f, 0.0f, 0.0f));
    v3 pw = xform_point(c.m, V(x_ndc, y_ndc, c.fov_dist));
    d = normalize(pw - o);
}

// ---- closest / any hit over the flattened BVH -----------------------------------------------------------------------------
struct Hit
{
    float t;      // -1 = none (hit_info.h:11)
    int prim;     // original primitive index
    int slot;     // slot in the leaf-ordered triangle stream (-1 for spheres)
    float u, v;
    v3 sphere_n;  // only meaningful when slot < 0 && prim >= 0
};

enum TraceMode { TRACE_CLOSEST = 0, TRACE_ANY = 1, TRACE_SHADOW = 2 };

struct RaySlabs
{
    float ix, iy, iz;        // clamped reciprocals of the direction
    float ox, oy, oz;        // origin * reciprocal: slab distance = fma(plane, i, -o) (one FFMA; conservative within the builder's pad)
    float rc[4], na[4], nb[4];
};

__device__ __forceinline__ float safe_rcp(float d)
{
    return 1.0f / (fabsf(d) < 1e-30f ? copysignf(1e-30f, d) : d);
}

__device__ __forceinline__ void setup_slabs(v3 o, v3 d, bool use_diag, RaySlabs& rs)
{
    rs.ix = safe_rcp(d.x); rs.iy = safe_rcp(d.y); rs.iz = safe_rcp(d.z);
    rs.ox = o.x * rs.ix; rs.oy = o.y * rs.iy; rs.oz = o.z * rs.iz;
    if (use_diag)
    {
        // diagonal planes (+-1, +-1, 1) (the reference's PLANE_NORMALS[3..6] without the common sqrt(3)/3, bvh.cpp:8-16)
        const float d1 = fabsf(d.x) + fabsf(d.y) + fabsf(d.z);
        const float slack = 2.384185791015625e-07f * (fabsf(o.x) + fabsf(o.y) + fabsf(o.z));   // 2^-22 |o|_1 bounds numer rounding
        const float den[4] = { (d.x + d.y) + d.z, (-d.x + d.y) + d.z, (-d.x - d.y) + d.z, (d.x - d.y) + d.z };
        const float num[4] = { (o.x + o.y) + o.z, (-o.x + o.y) + o.z, (-o.x - o.y) + o.z, (o.x - o.y) + o.z };
#pragma unroll
        for (int k = 0; k < 4; k++)
        {
            // near-parallel planes are switched off: their reciprocal is too inexact to stay conservative
            bool on = fabsf(den[k]) >= 0.03f * d1;
            rs.rc[k] = on ? 1.0f / den[k] : 1.0f;
            rs.na[k] = on ? num[k] + slack : 1e30f;
            rs.nb[k] = on ? num[k] - slack : -1e30f;
        }
    }
}

// Möller–Trumbore exactly as include/triangle.h:16-60, on the stored a, e1 = b - a, e2 = c - a
__device__ __forceinline__ bool tri_test(const float4 va, const float4 ve1, const float4 ve2, v3 o, v3 d, float& t_out, float& u_out, float& v_out)
{
    const float EPSILON = 0.0000001f;
    v3 edge1 = V(ve1.x, ve1.y, ve1.z), edge2 = V(ve2.x, ve2.y, ve2.z);
    v3 h = cross(d, edge2);
    float a = dot(edge1, h);
    if (a > -EPSILON && a < EPSILON) return false;
    float f = 1.0f / a;
    v3 s = o - V(va.x, va.y, va.z);
    float u = f * dot(s, h);
    if (u < 0.0f || u > 1.0f) return false;
    v3 q = cross(s, edge1);
    float v = f * dot(d, q);
    if (v < 0.0f || u + v > 1.0f) return false;
    float t = f * dot(edge2, q);
    if (t > EPSILON) { t_out = t; u_out = u; v_out = v; return true; }
    return false;
}

// Traversal state of one ray. MODE:
//   TRACE_CLOSEST : exact closest hit over all triangles (== brute force, ties -> lowest index)
//   TRACE_ANY     : any triangle hit with t > EPSILON                       (occlusion test of render_kernel.cpp:592,:615)
//   TRACE_SHADOW  : any triangle hit with t + 1e-4f < tmax                  (evaluate_shadow_ray, :744-759)
// MODE is a run-time value so that one copy of the loop serves every ray type of the integrators' single trace site
// (it is only consulted when a triangle test succeeds). The state is explicit so that the same step function serves
// the run-to-completion traversal (megakernel, primary rays) and the persistent trace kernel that refills idle lanes
// with new rays between steps.
struct Trav
{
    v3 o, d;
    float tmax, tbest;
    int mode, cur, sp;
    bool done;
    RaySlabs rs;
    Hit hit;
};
// the per-lane traversal stack lives in local memory, outside Trav, so the rest of the state stays in registers
struct TravStack
{
    int ref[kStackSize];
    float t[kStackSize];
};

template <bool use_diag>
__device__ __forceinline__ void trav_init(Trav& T, v3 o, v3 d, float tmax, const int mode)
{
    T.o = o; T.d = d; T.tmax = tmax; T.mode = mode;
    setup_slabs(o, d, use_diag, T.rs);
    T.tbest = (mode == TRACE_SHADOW) ? tmax : __int_as_float(0x7f800000);
    T.hit.t = -1.0f; T.hit.prim = -1; T.hit.slot = -1;
    T.sp = 0; T.cur = 0; T.done = false;
}

// pop the next subtree, skipping those that start beyond the current best; T.done when the stack is empty
__device__ __forceinline__ void trav_pop(Trav& T, TravStack& K)
{
    for (;;)
    {
        if (T.sp == 0) { T.done = true; return; }
        T.sp--;
        if (K.t[T.sp] <= T.tbest * 1.00004f) { T.cur = K.ref[T.sp]; return; }
    }
}

// visit the inner node T.cur (>= 0): test both children, descend into the nearer hit one (pushing the other) or pop
template <bool use_diag>
__device__ __forceinline__ void trav_inner(const SceneDev& S, Trav& T, TravStack& K)
{

    const RaySlabs& rs = T.rs;
    const float tbest = T.tbest;
    {
        const float4* an = S.axis + 4 * (size_t)T.cur;
        const float4 n0 = __ldg(an + 0), n1 = __ldg(an + 1), n2 = __ldg(an + 2), n3 = __ldg(an + 3);
        // L: lo = (n0.x n0.y n0.z) hi = (n0.w n1.x n1.y); R: lo = (n1.z n1.w n2.x) hi = (n2.y n2.z n2.w)
        // The slab distances only have to be conservative (the exact test is Moller-Trumbore): one fused multiply-add each.
        // Rounding moves a plane by at most ~2^-23 |o| along its axis, inside the pad the builder put around every volume.
        float a0 = fmaf(n0.x, rs.ix, -rs.ox), a1 = fmaf(n0.w, rs.ix, -rs.ox);
        float b0 = fmaf(n0.y, rs.iy, -rs.oy), b1 = fmaf(n1.x, rs.iy, -rs.oy);
        float c0 = fmaf(n0.z, rs.iz, -rs.oz), c1 = fmaf(n1.y, rs.iz, -rs.oz);
        float tnL = fmaxf(fmaxf(fminf(a0, a1), fminf(b0, b1)), fmaxf(fminf(c0, c1), 0.0f));
        float tfL = fminf(fminf(fmaxf(a0, a1), fmaxf(b0, b1)), fminf(fmaxf(c0, c1), tbest));
        a0 = fmaf(n1.z, rs.ix, -rs.ox); a1 = fmaf(n2.y, rs.ix, -rs.ox);
        b0 = fmaf(n1.w, rs.iy, -rs.oy); b1 = fmaf(n2.z, rs.iy, -rs.oy);
        c0 = fmaf(n2.x, rs.iz, -rs.oz); c1 = fmaf(n2.w, rs.iz, -rs.oz);
        float tnR = fmaxf(fmaxf(fminf(a0, a1), fminf(b0, b1)), fmaxf(fminf(c0, c1), 0.0f));
        float tfR = fminf(fminf(fmaxf(a0, a1), fmaxf(b0, b1)), fminf(fmaxf(c0, c1), tbest));
        // distance-proportional widening keeps the float slab test conservative (Ize, "Robust BVH ray traversal")
        bool hitL = tnL <= tfL * 1.000001f;
        bool hitR = tnR <= tfR * 1.000001f;
        if (use_diag && (hitL || hitR))
        {
            const float4* dn = S.diag + 4 * (size_t)T.cur;
            if (hitL)
            {
                const float4 nr = __ldg(dn + 0), fr = __ldg(dn + 1);
                float p0 = (nr.x - rs.na[0]) * rs.rc[0], q0 = (fr.x - rs.nb[0]) * rs.rc[0];
                float p1 = (nr.y - rs.na[1]) * rs.rc[1], q1 = (fr.y - rs.nb[1]) * rs.rc[1];
                float p2 = (nr.z - rs.na[2]) * rs.rc[2], q2 = (fr.z - rs.nb[2]) * rs.rc[2];
                float p3 = (nr.w - rs.na[3]) * rs.rc[3], q3 = (fr.w - rs.nb[3]) * rs.rc[3];
                float tn = fmaxf(fmaxf(fminf(p0, q0), fminf(p1, q1)), fmaxf(fminf(p2, q2), fminf(p3, q3)));
                float tf = fminf(fminf(fmaxf(p0, q0), fmaxf(p1, q1)), fminf(fmaxf(p2, q2), fmaxf(p3, q3)));
                tnL = fmaxf(tnL, tn); tfL = fminf(tfL, tf);
                hitL = tnL <= tfL * 1.00004f;
            }
            if (hitR)
            {
                const float4 nr = __ldg(dn + 2), fr = __ldg(dn + 3);
                float p0 = (nr.x - rs.na[0]) * rs.rc[0], q0 = (fr.x - rs.nb[0]) * rs.rc[0];
                float p1 = (nr.y - rs.na[1]) * rs.rc[1], q1 = (fr.y - rs.nb[1]) * rs.rc[1];
                float p2 = (nr.z - rs.na[2]) * rs.rc[2], q2 = (fr.z - rs.nb[2]) * rs.rc[2];
                float p3 = (nr.w - rs.na[3]) * rs.rc[3], q3 = (fr.w - rs.nb[3]) * rs.rc[3];
                float tn = fmaxf(fmaxf(fminf(p0, q0), fminf(p1, q1)), fmaxf(fminf(p2, q2), fminf(p3, q3)));
                float tf = fminf(fminf(fmaxf(p0, q0), fmaxf(p1, q1)), fminf(fmaxf(p2, q2), fmaxf(p3, q3)));
                tnR = fmaxf(tnR, tn); tfR = fminf(tfR, tf);
                hitR = tnR <= tfR * 1.00004f;
            }
        }
        const int refL = __float_as_int(n3.x), refR = __float_as_int(n3.y);
        if (hitL && hitR)
        {
            const bool r_first = tnR < tnL;
            K.ref[T.sp] = r_first ? refL : refR;
            K.t[T.sp] = r_first ? tnL : tnR;
            T.sp++;
            T.cur = r_first ? refR : refL;
            return;
        }
        if (hitL) { T.cur = refL; return; }
        if (hitR) { T.cur = refR; return; }
    }
    trav_pop(T, K);
}

// visit the leaf T.cur (< 0): exact triangle tests, then pop
__device__ __forceinline__ void trav_leaf(const SceneDev& S, Trav& T, TravStack& K)
{
    const v3 o = T.o, d = T.d;
    {
        const int packed = ~T.cur;
        const int first = packed >> 4, count = packed & 15;
        const float4* tp = S.tris + 3 * (size_t)first;
        for (int i = 0; i < count; i++, tp += 3)
        {
            const float4 va = __ldg(tp), ve1 = __ldg(tp + 1), ve2 = __ldg(tp + 2);
            float t, u, v;
            if (tri_test(va, ve1, ve2, o, d, t, u, v))
            {
                if (T.mode == TRACE_ANY) { T.hit.t = t; T.done = true; return; }
                if (T.mode == TRACE_SHADOW) { if (t + 1.0e-4f < T.tmax) { T.hit.t = t; T.done = true; return; } continue; }
                const int prim = __float_as_int(va.w);
                // strict "<" (bvh.h:158); equal t goes to the lower original index, as brute force would (render_kernel.cpp:464)
                if (T.hit.prim < 0 || t < T.hit.t || (t == T.hit.t && prim < T.hit.prim))
                {
                    T.hit.t = t; T.hit.prim = prim; T.hit.slot = first + i; T.hit.u = u; T.hit.v = v;
                    T.tbest = t;
                }
            }
        }
    }
    trav_pop(T, K);
}

// one step of either kind (the persistent trace kernel advances lanes step by step)
template <bool use_diag>
__device__ __forceinline__ void trav_step(const SceneDev& S, Trav& T, TravStack& K)
{
    if (T.cur >= 0) trav_inner<use_diag>(S, T, K);
    else trav_leaf(S, T, K);
}

// Returns true when a hit was found (see Trav for MODE). "while-while": every lane descends through inner nodes until
// it holds a leaf (or is finished); the lanes of a warp reconverge at the end of that inner loop, so the expensive
// exact triangle tests run with as many lanes as possible instead of interleaving with other lanes' node tests.
template <bool use_diag>
__device__ __forceinline__ bool traverse_tris(const SceneDev& S, v3 o, v3 d, float tmax, const int MODE, Hit& hit)
{
    Trav T;
    TravStack K;
    trav_init<use_diag>(T, o, d, tmax, MODE);
    while (!T.done)
    {
        while (T.cur >= 0 && !T.done) trav_inner<use_diag>(S, T, K);
        if (T.done) break;
        trav_leaf(S, T, K);
    }
    hit = T.hit;
    return hit.t > 0.0f;
}

// ---- wide (8-ary, quantised) BVH ----------------------------------------------------------------------------------------------
// The default acceleration structure on the device: 80-byte nodes (5 x LDG.128) holding 8 children whose boxes are
// quantised to one byte per plane relative to the node's own frame (after Ylitie, Karras, Laine, "Efficient incoherent ray
// traversal on GPUs through compressed wide BVHs", HPG 2017, re-encoded for this machine). One node fetch advances a
// ray three binary levels, so the dependent fetch chain that bounds a trace pass is ~3x shorter than with the binary
// layout above and a ray touches ~3x fewer bytes. Layout (host twin: WideNode in bvh_build.h):
//   n0 = { p.x, p.y, p.z, [ex | ey << 8 | ez << 16 | imask << 24] }   frame origin, per-axis cell size 2^(e - 127), inner-child mask by slot
//   n1 = { child_base, tri_base, valid24, 0 }                           first inner child (node index), first triangle slot, triangle map
//   n2 = { lox[0..3], lox[4..7], loy[0..3], loy[4..7] }  n3 = { loz, loz, hix, hix }  n4 = { hiy, hiy, hiz, hiz }
// A plane byte q decodes — with ONE byte permute, no int->float conversion — to the float whose bits are
// 0x43000000 | q << 16, i.e. v(q) = 128 + q for q < 128 and 2q for q >= 128: a monotone 256-level grid over
// [128, 510] cells (fine near the frame origin, twice as coarse beyond). plane = p + 2^e * v(q); the builder rounds
// lo planes down and hi planes up on that grid, so a decoded box always contains the padded float box.
// valid24: bit 3s + i set = slot s is a leaf child holding a triangle i (at most 3); the node's triangles are stored
// compactly from tri_base in that bit order, so triangle (s, i) is at tri_base + popc(valid24 below bit 3s + i).
// Children sit in the slot whose octant (bit a set = positive side of axis a) best matches their position, so that
// "slot ^ (7 - ray octant)" orders them front to back for any ray direction.
struct Trav8
{
    v3 o, d;
    float tmax, tbest;
    int mode, sp;
    bool done;
    float ix, iy, iz;          // clamped reciprocals of the direction
    unsigned int oct;          // 7 - ray octant
    uint2 ng;                  // node group: x = index of the first inner child, y = hit bits (24..31, front-to-back order) | imask
    uint2 tg;                  // triangle group: x = first triangle slot of the node, y = hit bits in valid24 positions
    unsigned int tvalid;       // valid24 of the node the triangle group belongs to
    Hit hit;
};
// Stack of node groups. TravStack8: per-lane local memory (lane-interleaved 4-byte words: lanes at different depths touch a
// different 32-byte sector each, 2.5 useful bytes per sector in ncu, local-load L1 hit rate 54 % in wf_trace_coop).
// TravStack8Shared: the first kSharedStackDepth entries (a C3 tree is 9 levels deep, the 20 M-triangle tree 12) in shared
// memory, one 8-byte column per thread, the rest in local memory.
struct TravStack8
{
    uint2 e[kStackSize];
    __device__ __forceinline__ void push(int sp, uint2 v) { e[sp] = v; }
    __device__ __forceinline__ uint2 pop(int sp) const { return e[sp]; }
};
constexpr int kSharedStackDepth = 10;
struct TravStack8Shared
{
    uint2* sh;          // this thread's column: entry i at sh[i * blockDim.x]
    int stride;
    uint2 ovf[kStackSize - kSharedStackDepth];
    __device__ __forceinline__ void push(int sp, uint2 v) { if (sp < kSharedStackDepth) sh[sp * stride] = v; else ovf[sp - kSharedStackDepth] = v; }
    __device__ __forceinline__ uint2 pop(int sp) const { return sp < kSharedStackDepth ? sh[sp * stride] : ovf[sp - kSharedStackDepth]; }
};

__device__ __forceinline__ float safe_rcp8(float d)
{
    return 1.0f / (fabsf(d) < 1e-20f ? copysignf(1e-20f, d) : d);
}

__device__ __forceinline__ void trav8_init(Trav8& T, v3 o, v3 d, float tmax, const int mode)
{
    T.o = o; T.d = d; T.tmax = tmax; T.mode = mode;
    T.ix = safe_rcp8(d.x); T.iy = safe_rcp8(d.y); T.iz = safe_rcp8(d.z);
    T.oct = 7u - ((T.ix < 0.0f ? 1u : 0u) | (T.iy < 0.0f ? 2u : 0u) | (T.iz < 0.0f ? 4u : 0u));
    T.tbest = (mode == TRACE_SHADOW) ? tmax : __int_as_float(0x7f800000);
    T.hit.t = -1.0f; T.hit.prim = -1; T.hit.slot = -1;
    T.sp = 0; T.done = false;
    T.ng = make_uint2(0u, 0x80000000u);      // the root as the only member of a node group with an empty imask
    T.tg = make_uint2(0u, 0u);
    T.tvalid = 0u;
}

__device__ __forceinline__ bool trav8_has_node(const Trav8& T) { return T.tg.y == 0u; }     // else: triangles pending

template <typename Stack>
__device__ __forceinline__ void trav8_pop(Trav8& T, Stack& K)
{
    if (T.sp == 0) { T.done = true; return; }
    T.ng = K.pop(--T.sp);
}

// slot of the triangle behind bit b of a triangle group
__device__ __forceinline__ int trav8_tri_slot(const Trav8& T, int b) { return (int)(T.tg.x + __popc(T.tvalid & ((1u << b) - 1u))); }

// plane byte j of w -> float v(q) (see above). The constant 0x43000000 comes from the kernel's parameter block, opaque to
// ptxas, so that it lives in a register and the selector can be the PRMT's immediate; otherwise every PRMT needs an
// extra move of its selector into a register.
#define B200RT_Q(w, j) __uint_as_float(__byte_perm((w), qmagic, 0x7044u | ((j) << 8)))

// Tests child j (bytes j of the near / far plane words) and shifts its miss bit (the sign of t_far * (1 + 2^-20) - t_near:
// distance-proportional widening keeps the float slab test conservative, Ize; the boxes themselves are padded by the
// builder) into acc. One funnel shift instead of compare + select + shift + or. A NaN counts as a hit.
#define B200RT_WIDE_CHILD(j)                                                                                                   \
    {                                                                                                                          \
        const float tnx = fmaf(B200RT_Q(nx, j), sx, ox), tfx = fmaf(B200RT_Q(fx, j), sx, ox);                                  \
        const float tny = fmaf(B200RT_Q(ny, j), sy, oy), tfy = fmaf(B200RT_Q(fy, j), sy, oy);                                  \
        const float tnz = fmaf(B200RT_Q(nz, j), sz, oz), tfz = fmaf(B200RT_Q(fz, j), sz, oz);                                  \
        const float tn = fmaxf(fmaxf(tnx, tny), fmaxf(tnz, 0.0f));                                                             \
        const float tf = fminf(fminf(tfx, tfy), fminf(tfz, tbest));                                                            \
        acc = __funnelshift_l(__float_as_uint(fmaf(tf, 1.000001f, -tn)), acc, 1);                                              \
    }

// children 3, 2, 1, 0 of one half, in that order (child j of the node ends up at bit j of ~acc)
__device__ __forceinline__ unsigned int wide_test4(unsigned int acc, unsigned int nx, unsigned int fx, unsigned int ny, unsigned int fy,
                                                   unsigned int nz, unsigned int fz, float sx, float sy, float sz, float ox, float oy,
                                                   float oz, float tbest, unsigned int qmagic)
{
    B200RT_WIDE_CHILD(3) B200RT_WIDE_CHILD(2) B200RT_WIDE_CHILD(1) B200RT_WIDE_CHILD(0)
    return acc;
}

// pre: trav8_has_node(T) and the node group holds at least one hit. Takes the front-most child node of the group, tests
// its 8 children, leaves the hit inner children in T.ng and the hit triangles in T.tg.
template <typename Stack>
__device__ __forceinline__ void trav8_node(const SceneDev& S, Trav8& T, Stack& K)
{
    const unsigned int hits = T.ng.y;
    const int bit = 31 - __clz((int)hits);
    T.ng.y = hits & ~(1u << bit);
    if (T.ng.y & 0xff000000u) K.push(T.sp++, T.ng);        // the group's remaining members wait on the stack
    const unsigned int slot = (unsigned int)(bit - 24) ^ T.oct;
    const unsigned int rel = __popc(hits & 0xffu & ~(0xffffffffu << slot));
    const float4* np = S.wide + 5 * (size_t)(T.ng.x + rel);
    const float4 n0 = __ldg(np), n1 = __ldg(np + 1), n2 = __ldg(np + 2), n3 = __ldg(np + 3), n4 = __ldg(np + 4);
    const unsigned int ew = __float_as_uint(n0.w);
    const float sx = __uint_as_float((ew & 0xffu) << 23) * T.ix;
    const float sy = __uint_as_float(((ew >> 8) & 0xffu) << 23) * T.iy;
    const float sz = __uint_as_float(((ew >> 16) & 0xffu) << 23) * T.iz;
    const float ox = (n0.x - T.o.x) * T.ix, oy = (n0.y - T.o.y) * T.iy, oz = (n0.z - T.o.z) * T.iz;
    const bool bx = T.ix < 0.0f, by = T.iy < 0.0f, bz = T.iz < 0.0f;
    const unsigned int lox0 = __float_as_uint(n2.x), lox1 = __float_as_uint(n2.y), loy0 = __float_as_uint(n2.z), loy1 = __float_as_uint(n2.w);
    const unsigned int loz0 = __float_as_uint(n3.x), loz1 = __float_as_uint(n3.y), hix0 = __float_as_uint(n3.z), hix1 = __float_as_uint(n3.w);
    const unsigned int hiy0 = __float_as_uint(n4.x), hiy1 = __float_as_uint(n4.y), hiz0 = __float_as_uint(n4.z), hiz1 = __float_as_uint(n4.w);
    const unsigned int qmagic = S.qmagic;
    unsigned int acc = wide_test4(0u, bx ? hix1 : lox1, bx ? lox1 : hix1, by ? hiy1 : loy1, by ? loy1 : hiy1, bz ? hiz1 : loz1, bz ? loz1 : hiz1,
                                  sx, sy, sz, ox, oy, oz, T.tbest, qmagic);
    acc = wide_test4(acc, bx ? hix0 : lox0, bx ? lox0 : hix0, by ? hiy0 : loy0, by ? loy0 : hiy0, bz ? hiz0 : loz0, bz ? loz0 : hiz0,
                     sx, sy, sz, ox, oy, oz, T.tbest, qmagic);
    const unsigned int imask = ew >> 24;
    const unsigned int hit8 = ~acc & 0xffu;                // bit s: the box in slot s is hit (empty slots are filtered by imask / valid24)
    // inner children: reorder the hit bits front to back for this ray's octant (bit s -> bit s ^ oct) with a 2 KB table
    const unsigned int inner = __ldg(S.oct_lut + ((T.oct << 8) | (hit8 & imask)));
    // leaf children: spread bit s to bits 3s..3s+2 (multiplies stand in for shift-or: the operands never overlap) and keep the real triangles
    unsigned int x = hit8 & ~imask;
    x = (x * 0x101u) & 0x0000f00fu;
    x = (x * 0x11u) & 0x000c30c3u;
    x = (x * 0x5u) & 0x00249249u;
    T.tvalid = __float_as_uint(n1.z);
    T.ng.x = __float_as_uint(n1.x);
    T.ng.y = (inner << 24) | imask;
    T.tg.x = __float_as_uint(n1.y);
    T.tg.y = (x * 7u) & T.tvalid;
    if (T.tg.y == 0u && !inner) trav8_pop(T, K);
}

// pre: !trav8_has_node(T). Exact triangle tests of the pending triangle group, then the next node group.
template <typename Stack>
__device__ __forceinline__ void trav8_tris(const SceneDev& S, Trav8& T, Stack& K)
{
    const v3 o = T.o, d = T.d;
    unsigned int bits = T.tg.y;
    T.tg.y = 0u;
    while (bits)
    {
        const int b = __ffs((int)bits) - 1;
        bits &= bits - 1u;
        const int slot = trav8_tri_slot(T, b);
        const float4* tp = S.tris + 3 * (size_t)slot;
        const float4 va = __ldg(tp), ve1 = __ldg(tp + 1), ve2 = __ldg(tp + 2);
        float t, u, v;
        if (tri_test(va, ve1, ve2, o, d, t, u, v))
        {
            if (T.mode == TRACE_ANY) { T.hit.t = t; T.done = true; return; }
            if (T.mode == TRACE_SHADOW) { if (t + 1.0e-4f < T.tmax) { T.hit.t = t; T.done = true; return; } continue; }
            const int prim = __float_as_int(va.w);
            // strict "<" (bvh.h:158); equal t goes to the lower original index, as brute force would (render_kernel.cpp:464)
            if (T.hit.prim < 0 || t < T.hit.t || (t == T.hit.t && prim < T.hit.prim))
            {
                T.hit.t = t; T.hit.prim = prim; T.hit.slot = slot; T.hit.u = u; T.hit.v = v;
                T.tbest = t;
            }
        }
    }
    if (!(T.ng.y & 0xff000000u)) trav8_pop(T, K);
}

__device__ __forceinline__ bool traverse_tris_wide(const SceneDev& S, v3 o, v3 d, float tmax, const int MODE, Hit& hit)
{
    Trav8 T;
    TravStack8 K;
    trav8_init(T, o, d, tmax, MODE);
    while (!T.done)
    {
        while (!T.done && trav8_has_node(T)) trav8_node(S, T, K);
        if (T.done) break;
        trav8_tris(S, T, K);
    }
    hit = T.hit;
    return hit.t > 0.0f;
}

// Sphere::intersect, include/sphere.h:11-53
__device__ __forceinline__ bool sphere_test(const SphereDev& s, v3 o, v3 d, float& t_out)
{
    v3 L = o - V(s.cx, s.cy, s.cz);
    float b = 2.0f * dot(d, L);
    float c = dot(L, L) - s.radius * s.radius;
    float delta = b * b - 4.0f * 1.0f * c;
    if (delta < 0.0f) return false;
    float t = -1.0f;
    if (delta == 0.0f) t = -b / 2.0f;
    else
    {
        float sq = sqrtf(delta);
        float t1 = (-b - sq) / 2.0f;
        float t2 = (-b + sq) / 2.0f;
        if (t1 < t2) { t = t1; if (t < 0.0f) t = t2; }
    }
    if (t < 0.0f) return false;
    t_out = t;
    return true;
}

// second half of INTERSECT_SCENE: every analytic sphere after the triangles (render_kernel.cpp:491-501)
__device__ __forceinline__ bool finish_with_spheres(const SceneDev& S, v3 o, v3 d, float tmax, const int mode, Hit& hit)
{
    for (int i = 0; i < S.n_spheres; i++)
    {
        float t;
        const SphereDev s = S.spheres[i];
        if (sphere_test(s, o, d, t))
            if (t < hit.t || hit.t == -1.0f)
            {
                hit.t = t; hit.prim = s.prim; hit.slot = -1; hit.u = -1.0f; hit.v = -1.0f;
                v3 p = o + t * d;
                hit.sphere_n = normalize(p - V(s.cx, s.cy, s.cz));
            }
    }
    bool found = hit.t > 0.0f;
    if (mode == TRACE_SHADOW) found = found && (hit.t + 1.0e-4f < tmax);
    return found;
}

// INTERSECT_SCENE (render_kernel.cpp:485-511): BVH triangles, then every analytic sphere; "found" iff closest.t > 0.
// mode TRACE_ANY / TRACE_SHADOW return the occlusion predicates of :592/:615 and evaluate_shadow_ray (:744-759).
// With analytic spheres in the scene the exact "closest.t > 0" semantics need the true closest hit (a sphere can
// report t == 0), so the early-out traversals are only used for triangle-only scenes.
// traversal layouts a kernel can be instantiated for
enum TravLayout { TL_AXIS = 0, TL_DIAG = 1, TL_WIDE = 2 };

template <int TL>
__device__ __forceinline__ bool traverse_any_layout(const SceneDev& S, v3 o, v3 d, float tmax, const int mode, Hit& hit)
{
    if constexpr (TL == TL_WIDE) return traverse_tris_wide(S, o, d, tmax, mode, hit);
    else return traverse_tris<TL == TL_DIAG>(S, o, d, tmax, mode, hit);
}

template <int TL>
__device__ __forceinline__ bool trace_ray(const SceneDev& S, v3 o, v3 d, float tmax, const int mode, Hit& hit)
{
    if (S.n_spheres == 0) return traverse_any_layout<TL>(S, o, d, tmax, mode, hit);
    traverse_any_layout<TL>(S, o, d, tmax, TRACE_CLOSEST, hit);
    return finish_with_spheres(S, o, d, tmax, mode, hit);
}

// point and geometric normal of a closest hit (triangle.h:46-49: normalize(cross(e1,e2)), never flipped)
__device__ __forceinline__ void hit_geometry(const SceneDev& S, const Hit& hit, v3 o, v3 d, v3& p, v3& n)
{
    p = o + hit.t * d;
    if (hit.slot >= 0)
    {
        const float4 ve1 = __ldg(S.tris + 3 * (size_t)hit.slot + 1), ve2 = __ldg(S.tris + 3 * (size_t)hit.slot + 2);
        n = normalize(cross(V(ve1.x, ve1.y, ve1.z), V(ve2.x, ve2.y, ve2.z)));
    }
    else n = hit.sphere_n;
}

// ---- BRDF: render_kernel.cpp:5-22, :218-301, :392-451, :513-518 ---------------------------------------------------------------
__device__ __forceinline__ v3 rotate_around_normal(v3 n, v3 local)
{
    float sign = copysignf(1.0f, n.z);
    const float a = -1.0f / (sign + n.z);
    const float b = n.x * n.y * a;
    v3 b1 = V(1.0f + sign * n.x * n.x * a, sign * b, -sign * n.x);
    v3 b2 = V(b, sign + n.y * n.y * a, -n.y);
    return (local.x * b1 + local.y * b2) + local.z * n;
}
__device__ __forceinline__ float ggx_d(float alpha, float NoH)
{
    NoH = smin(NoH, 0.999999f);
    float alpha2 = alpha * alpha;
    float NoH2 = NoH * NoH;
    float b = (NoH2 * (alpha2 - 1.0f) + 1.0f);
    return (float)((double)alpha2 * B200RT_1_PI_D / (double)(b * b));      // evaluated in double by the reference (:232)
}
__device__ __forceinline__ float g1_schlick(float k, float dp) { return dp / (dp * (1.0f - k) + k); }
__device__ __forceinline__ float power_heuristic(float a, float b) { float a2 = a * a; return a2 / (a2 + b * b); }

// D = ggx_d(roughness^2, NoH), computed by the caller (the light- and env-sample paths need it for the pdf whether or not the BRDF
// itself is evaluated: one double-precision division per pair instead of two)
__device__ __forceinline__ col ct_terms(const MaterialDev& m, float NoV, float NoL, float NoH, float VoH, float D, float* pdf_out)   // :272-298 / :424-448
{
    const float metalness = m.metalness;
    const float alpha = m.roughness * m.roughness;
    const float f04 = 0.04f * (1.0f - metalness);
    const col F0 = CO(f04 + m.dr * metalness, f04 + m.dg * metalness, f04 + m.db * metalness);
    // pow(1 - VoH, 5.0f) (:219): three double multiplications and one rounding — the correctly rounded value in all but ~1e-9 of the
    // cases, which is what glibc's powf returns to the reference; CUDA's powf is a 70-instruction routine (9.4 % of the shading step's
    // instructions, five evaluations per surface interaction) that is off by one ulp in 3 % of the cases
    const double omv = (double)(1.0f - VoH);
    const double omv2 = omv * omv;
    const float p5 = (float)((omv2 * omv2) * omv);
    const col F = CO(F0.r + (1.0f + -F0.r) * p5, F0.g + (1.0f + -F0.g) * p5, F0.b + (1.0f + -F0.b) * p5);   // fresnel_schlick :218-221
    const float k = alpha / 2.0f;
    const float G = g1_schlick(k, NoL) * g1_schlick(k, NoV);                                               // :240-245
    const float kd0 = 1.0f - metalness;
    const col kD = CO(kd0 * (1.0f + -F.r), kd0 * (1.0f + -F.g), kd0 * (1.0f + -F.b));
    const col diffuse_part = (kD * CO(m.dr, m.dg, m.db)) / B200RT_PI_F;
    const col specular_part = ((F * D) * G) / (4.0f * NoV * NoL);
    if (pdf_out) *pdf_out = D * NoH / (4.0f * VoH);
    return diffuse_part + specular_part;
}

// cook_torrance_brdf (:260-301) and cook_torrance_brdf_pdf (:247-258) of the same pair of directions, as sample_light_sources and
// sample_environment_map call them one after the other: the half vector, its two cosines and D are the same values in both
__device__ __forceinline__ col ct_brdf_and_pdf(const MaterialDev& m, v3 to_light, v3 view, v3 n, float& pdf)
{
    v3 h = normalize(view + to_light);
    float NoV = smax(0.0f, dot(n, view));
    float NoL = smax(0.0f, dot(n, to_light));
    float NoH = smax(0.0f, dot(n, h));
    float VoH = smax(0.0f, dot(h, view));
    const float D = ggx_d(m.roughness * m.roughness, NoH);
    pdf = D * NoH / (4.0f * VoH);
    if (NoV > 0.0f && NoL > 0.0f && NoH > 0.0f) return ct_terms(m, NoV, NoL, NoH, VoH, D, nullptr);
    return CO(0.0f, 0.0f, 0.0f);
}

// cook_torrance_brdf_importance_sample :392-451 — consumes exactly two draws
__device__ __forceinline__ col ct_sample(const MaterialDev& m, v3 view, v3 n, v3& out_dir, float& pdf, uint32_t& rng)
{
    pdf = 0.0f;
    const float alpha = m.roughness * m.roughness;
    const float rand1 = xs_float(rng);
    const float rand2 = xs_float(rng);
    const float phi = 2.0f * B200RT_PI_F * rand1;
    const float theta = acosf((1.0f - rand2) / (rand2 * (alpha * alpha - 1.0f) + 1.0f));   // no sqrt: the reference's own variant (:404)
    // sincosf returns exactly sinf / cosf of the argument (checked on 1e8 arguments in [0, 2 pi]: no differing bit) for one range
    // reduction instead of two
    float sin_theta, cos_theta, sin_phi, cos_phi;
    sincosf(theta, &sin_theta, &cos_theta);
    sincosf(phi, &sin_phi, &cos_phi);
    v3 local = V(cos_phi * sin_theta, sin_phi * sin_theta, cos_theta);
    v3 mn = rotate_around_normal(n, local);
    if (dot(mn, n) < 0.0f) return CO(0.0f, 0.0f, 0.0f);
    v3 to_light = normalize((2.0f * dot(mn, view)) * mn - view);
    out_dir = to_light;
    float NoV = smax(0.0f, dot(n, view));
    float NoL = smax(0.0f, dot(n, to_light));
    float NoH = smax(0.0f, dot(n, mn));
    float VoH = smax(0.0f, dot(mn, view));
    if (NoV > 0.0f && NoL > 0.0f && NoH > 0.0f) return ct_terms(m, NoV, NoL, NoH, VoH, ggx_d(alpha, NoH), &pdf);
    return CO(0.0f, 0.0f, 0.0f);
}

// ---- environment map: render_kernel.cpp:520-567, image.h:80-85,:165-177 ------------------------------------------------------
__device__ __forceinline__ col env_texel(const SceneDev& S, int idx) { float4 p = __ldg(S.env + idx); return CO(p.x, p.y, p.z); }
__device__ __forceinline__ int env_offset(const SceneDev& S, int x, int y)
{
    int px = min(max(x, 0), S.env_w - 1), py = min(max(y, 0), S.env_h - 1);
    return py * S.env_w + px;
}
__device__ __forceinline__ col env_from_direction(const SceneDev& S, v3 d)
{
    float u = 0.5f + atan2f(d.z, d.x) / (2.0f * B200RT_PI_F);
    float v = 0.5f + asinf(d.y) / B200RT_PI_F;
    int x = max(min((int)(u * (float)S.env_w), S.env_w - 1), 0);
    int y = max(min((int)(v * (float)S.env_h), S.env_h - 1), 0);
    return env_texel(S, y * S.env_w + x);
}
__device__ __forceinline__ void env_cdf_search(const SceneDev& S, float value, int& xo, int& yo)
{
    if (S.cdf_guide)
    {
        // The reference's two binary searches (row on the last column, then column inside the row, :532-567) return the first texel
        // whose running sum exceeds `value` in row-major order (the last texel if none does) whenever the running sum is
        // non-decreasing — which env_tables.cu verified before it built this guide. The guide brackets that texel per value bucket
        // (~2 probes instead of 21 dependent ones on the 2048x1024 sky); the bracketed search returns the same texel, bit for bit.
        const unsigned int b = min((unsigned int)(S.cdf_guide_n - 1), __float2uint_rz(value * S.cdf_guide_scale));
        const unsigned int n_texels = (unsigned int)(S.env_w * S.env_h);
        unsigned int lower = __ldg(S.cdf_guide + b), upper = min(__ldg(S.cdf_guide + b + 2), n_texels - 1u);
        while (lower < upper)
        {
            const unsigned int mid = (lower + upper) >> 1;
            if (value < __ldg(S.cdf + mid)) upper = mid; else lower = mid + 1u;
        }
        yo = (int)(lower / (unsigned int)S.env_w);
        xo = (int)(lower - (unsigned int)yo * (unsigned int)S.env_w);
        return;
    }
    int lower = 0, upper = S.env_h - 1;
    while (lower < upper)
    {
        int y_index = (lower + upper) / 2;
        // same probes as the reference (cdf[y_index * W + W - 1], :541-547), read from a compact copy of that column
        if (value < __ldg(S.row_cdf + y_index)) upper = y_index; else lower = y_index + 1;
    }
    const int y = max(min(lower, S.env_h), 0);
    lower = 0; upper = S.env_w - 1;
    while (lower < upper)
    {
        int xi = (lower + upper) / 2;
        if (value < __ldg(S.cdf + y * S.env_w + xi)) upper = xi; else lower = xi + 1;
    }
    xo = max(min(lower, S.env_w), 0); yo = y;
}

// ---- one surface interaction, split into the reference's four "side rays" + the continuation ---------------------------------
// The RNG draw schedule per hit is fixed (SURVEY a5): [3 light] 2 | 1 2 | 2, and no draw depends on a trace result, so a
// hit is processed as: for k in 0..3 { generate side ray k; trace it; keep its contribution }, then the continuation.
struct Surface
{
    v3 p, n, view;       // hit point, geometric normal, -ray.direction
    MaterialDev m;
};

enum SideKind { SIDE_NONE = 0, SIDE_SHADOW = 1, SIDE_CLOSEST_LIGHT = 2, SIDE_OCCLUSION = 3 };

struct SideRay
{
    v3 o, d;
    float tmax;        // SIDE_SHADOW: distance to the light sample
    col weight;        // contribution if unoccluded (SIDE_CLOSEST_LIGHT: brdf * cosine, finished by side_light_hit)
    float pdf;         // SIDE_CLOSEST_LIGHT: direction pdf
    int kind;
};

// k = 0: light sample of sample_light_sources (:636-675, sample_random_point_on_lights :715-742); 3 draws iff emissive triangles exist
__device__ __forceinline__ void side_light_sample(const SceneDev& S, const Surface& sf, uint32_t& rng, SideRay& r)
{
    r.kind = SIDE_NONE;
    if (S.n_emissive <= 0) return;
    const int pick = (int)(xs_float(rng) * (float)S.n_emissive);
    const int em_tri = __ldg(S.emissive + pick);
    const float rand_1 = xs_float(rng);
    const float rand_2 = xs_float(rng);
    const int slot = __ldg(S.slot_of_prim + em_tri);
    const float4 va = __ldg(S.tris + 3 * (size_t)slot), ve1 = __ldg(S.tris + 3 * (size_t)slot + 1), ve2 = __ldg(S.tris + 3 * (size_t)slot + 2);
    const float sqrt_r1 = sqrtf(rand_1);
    const float u = 1.0f - sqrt_r1;
    const float v = (1.0f - rand_2) * sqrt_r1;
    const v3 AB = V(ve1.x, ve1.y, ve1.z), AC = V(ve2.x, ve2.y, ve2.z);
    const v3 lp = (V(va.x, va.y, va.z) + u * AB) + v * AC;
    const v3 nrm = cross(AB, AC);
    const float len_n = length(nrm);
    const v3 light_n = (1.0f / len_n) * nrm;
    const float area = len_n * 0.5f;
    float light_pdf = 1.0f / ((float)S.n_emissive * area);

    const v3 so = sf.p + 1.0e-4f * sf.n;
    const v3 sd = lp - so;
    const float dist = length(sd);
    const v3 sdn = normalize(sd);
    const float dot_light = smax(dot(light_n, -sdn), 0.0f);
    if (!(dot_light > 0.0f)) return;
    light_pdf *= dist * dist;
    light_pdf /= dot_light;
    float bp;
    const col brdf = ct_brdf_and_pdf(sf.m, sdn, sf.view, sf.n, bp);
    if (!(bp != 0.0f)) return;
    const MaterialDev em = S.mats[__ldg(S.mat_idx + em_tri)];
    const float w = power_heuristic(light_pdf, bp);
    const float cosine_term = dot(sf.n, sdn);
    r.weight = (((CO(em.er, em.eg, em.eb) * cosine_term) * brdf) * w) / light_pdf;     // :671
    r.o = so; r.d = sdn; r.tmax = dist; r.kind = SIDE_SHADOW;
}

// k = 1: BRDF sample of sample_light_sources (:677-710); 2 draws. The ray is a CLOSEST-hit query (it must know what it hit).
__device__ __forceinline__ void side_light_brdf(const SceneDev& S, const Surface& sf, uint32_t& rng, SideRay& r)
{
    r.kind = SIDE_NONE;
    v3 dir = V(0.0f, 0.0f, 0.0f);
    float pdf;
    const col brdf = ct_sample(sf.m, sf.view, sf.n, dir, pdf, rng);
    if (is_black(brdf)) return;
    r.o = sf.p + 1.0e-5f * sf.n; r.d = dir; r.pdf = pdf;
    r.weight = brdf * dot(sf.n, dir);      // (brdf * cosine_term) of :706
    r.kind = SIDE_CLOSEST_LIGHT;
}
// finishes k = 1 once the closest hit is known (:688-708)
__device__ __forceinline__ col side_light_hit(const SceneDev& S, const SideRay& r, const Hit& nh)
{
    v3 hp, hn;
    hit_geometry(S, nh, r.o, r.d, hp, hn);
    const float cos_angle = smax(dot(hn, -r.d), 0.0f);
    if (!(cos_angle > 0.0f)) return CO(0.0f, 0.0f, 0.0f);
    const MaterialDev hm = S.mats[__ldg(S.mat_idx + nh.prim)];
    if (!(hm.er > 0.0f || hm.eg > 0.0f || hm.eb > 0.0f)) return CO(0.0f, 0.0f, 0.0f);
    const float d2 = nh.t * nh.t;
    // Triangle::area (triangle.cpp:8-11); the reference indexes the triangle buffer with the primitive index, so an
    // emissive analytic sphere would read out of bounds there — spheres contribute no area light here.
    if (nh.slot < 0) return CO(0.0f, 0.0f, 0.0f);
    const float4 ve1 = __ldg(S.tris + 3 * (size_t)nh.slot + 1), ve2 = __ldg(S.tris + 3 * (size_t)nh.slot + 2);
    const float light_area = length(cross(V(ve1.x, ve1.y, ve1.z), V(ve2.x, ve2.y, ve2.z))) / 2.0f;
    const float light_pdf = d2 / (light_area * cos_angle);        // no 1/N_lights: kept (:702)
    const float w = power_heuristic(r.pdf, light_pdf);
    return ((r.weight * CO(hm.er, hm.eg, hm.eb)) * w) / r.pdf;
}

// k = 2: env-map sample of sample_environment_map (:571-604); 1 draw
__device__ __forceinline__ void side_env_sample(const SceneDev& S, const Surface& sf, uint32_t& rng, SideRay& r)
{
    r.kind = SIDE_NONE;
    const float total = S.cdf_total;
    int x, y;
    if (S.use_alias)
    {
        // the same single draw, taken as its 32 raw bits: texel = floor(r * N / 2^32), the low word of the product is the coin
        const unsigned int n_texels = (unsigned int)(S.env_w * S.env_h);
        const unsigned long long m = (unsigned long long)xs_next(rng) * n_texels;
        unsigned int i = (unsigned int)(m >> 32);
        const float2 a = __ldg(S.env_alias + i);
        if (!((float)(unsigned int)m * 2.3283064365386962890625e-10f < a.x)) i = (unsigned int)__float_as_int(a.y);
        y = (int)(i / (unsigned int)S.env_w); x = (int)(i - (unsigned int)y * (unsigned int)S.env_w);
    }
    else env_cdf_search(S, xs_float(rng) * total, x, y);
    const float u = (float)x / (float)S.env_w;
    const float v = (float)y / (float)S.env_h;
    const float phi = (float)((double)(u * 2.0f) * B200RT_PI_D);             // double in the reference (:578-579)
    const float theta = (float)((double)v * B200RT_PI_D);
    float sin_theta, cos_theta, sin_phi, cos_phi;
    sincosf(theta, &sin_theta, &cos_theta);
    sincosf(phi, &sin_phi, &cos_phi);
    const v3 dir = V(-sin_theta * cos_phi, -cos_theta, -sin_theta * sin_phi);
    const float cosine_term = dot(sf.n, dir);
    if (!(cosine_term > 0.0f)) return;
    const int idx = env_offset(S, x, y);
    const col radiance = env_texel(S, idx);
    float env_pdf = (float)(0.3086 * (double)radiance.r + 0.6094 * (double)radiance.g + 0.0820 * (double)radiance.b) / total;   // image.h:80-85
    env_pdf = (float)((double)((env_pdf * (float)S.env_w) * (float)S.env_h) / ((double)2.0f * B200RT_PI_D * B200RT_PI_D * (double)sin_theta));   // :595
    float brdf_pdf;
    const col brdf = ct_brdf_and_pdf(sf.m, dir, sf.view, sf.n, brdf_pdf);
    const float w = power_heuristic(env_pdf, brdf_pdf);
    r.weight = (((brdf * cosine_term) * w) * radiance) / env_pdf;          // :602
    r.o = sf.p + 1.0e-4f * sf.n; r.d = dir; r.kind = SIDE_OCCLUSION;
}

// k = 3: BRDF sample of sample_environment_map (:606-628); 2 draws
__device__ __forceinline__ void side_env_brdf(const SceneDev& S, const Surface& sf, uint32_t& rng, SideRay& r)
{
    r.kind = SIDE_NONE;
    v3 dir = V(0.0f, 0.0f, 0.0f);
    float bpdf;
    const col brdf = ct_sample(sf.m, sf.view, sf.n, dir, bpdf, rng);
    const float cosine_term = smax(dot(sf.n, dir), 0.0f);
    if (!(bpdf != 0.0f && cosine_term > 0.0f)) return;
    const col sky = env_from_direction(S, dir);
    const float theta_b = acosf(dir.z);                                     // z, not y: the reference's own convention (:618)
    const float sin_b = sinf(theta_b);
    float env_pdf = (0.3086f * sky.r + 0.6094f * sky.g + 0.0820f * sky.b) / S.cdf_total;
    env_pdf *= (float)(S.env_w * S.env_h);
    env_pdf = (float)((double)env_pdf / ((double)2.0f * B200RT_PI_D * B200RT_PI_D * (double)sin_b));
    const float w = power_heuristic(bpdf, env_pdf);
    r.weight = (((sky * w) * cosine_term) * brdf) / bpdf;                  // :626
    r.o = sf.p + 1.0e-5f * sf.n; r.d = dir; r.kind = SIDE_OCCLUSION;
}

// tone map of render_kernel.cpp:171-180 applied to (framebuffer + mean radiance); alpha follows the reference's Color ops
__device__ __forceinline__ float4 tonemap(float4 fb_in, col mean)
{
    const float gamma = 2.2f, exposure = 1.5f;
    const float r = fb_in.x + mean.r, g = fb_in.y + mean.g, b = fb_in.z + mean.b;
    float4 o;
    o.x = powf(1.0f + -expf(-r * exposure), 1.0f / gamma);
    o.y = powf(1.0f + -expf(-g * exposure), 1.0f / gamma);
    o.z = powf(1.0f + -expf(-b * exposure), 1.0f / gamma);
    o.w = 1.0f + -(-fb_in.w * exposure);      // Color::operator* scales alpha, exp()/pow() pass it through (color.h:149-183)
    return o;
}


// what a finished pixel writes into the tile buffer: the tone-mapped framebuffer value, or (B200RT_FLAG_LINEAR_TILES) the
// mean radiance itself, to be added to the framebuffer and tone-mapped by k_untile_accumulate on the gathering device
__device__ __forceinline__ float4 pixel_output(int flags, const float4* __restrict__ fb_in_rowmajor, size_t row_major_index, col mean)
{
    if (flags & B200RT_FLAG_LINEAR_TILES) return make_float4(mean.r, mean.g, mean.b, 0.0f);
    const float4 fb = fb_in_rowmajor ? fb_in_rowmajor[row_major_index] : make_float4(0.0f, 0.0f, 0.0f, 1.0f);
    return tonemap(fb, mean);
}

} // namespace b200rt
