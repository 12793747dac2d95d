// Device code shared by the device builder (bvh_build_gpu.cu lw_emit / lb_emit) and the refit (refit.cu): the per-axis pad of a child
// box, the leaf-ordered triangle record, and the choice of a wide node's frame with the outward quantisation of its child boxes. The
// refit calls the same functions the builder does, so a refitted node is what the builder would emit for the same child boxes.
#pragma once
#include <cfloat>
#include <cstdint>

#include <cuda_runtime.h>

#include "bvh_build.h"

namespace b200rt {

// the per-axis pad both layouts apply to a child box (device twin of box_pad in bvh_build.cpp)
__device__ __forceinline__ float box_pad_dev(float lo, float hi, float abs_pad) { return 1e-5f * fmaxf(fabsf(lo), fabsf(hi)) + abs_pad; }

// triangle `tri` of the original-order tri9 array as its leaf record: {a, as_float(tri)}, {b - a, 0}, {c - a, 0}
__device__ __forceinline__ void emit_triangle(const float* tri9, int tri, float4* out)
{
    const float* p = tri9 + 9 * (size_t)tri;
    out[0] = make_float4(p[0], p[1], p[2], __int_as_float(tri));
    out[1] = make_float4(p[3] - p[0], p[4] - p[1], p[5] - p[2], 0.0f);       // same float subtraction as triangle.h:21-22 / the host builder
    out[2] = make_float4(p[6] - p[0], p[7] - p[1], p[8] - p[2], 0.0f);
}

// Frame origin p, cell exponent e and the 8 x 2 plane bytes of every axis of `node` from the (already padded) child boxes klo / khi of
// the slots set in `used` (device twin of quantise_slots in bvh_build.cpp). Unused slots get inverted planes that are never hit. A box
// that does not fit the node's grid sets *overflow.
__device__ __forceinline__ void wide_quantise(WideNode& node, const float (&klo)[8][3], const float (&khi)[8][3], unsigned used, int* overflow)
{
    for (int a = 0; a < 3; a++)
    {
        float lo = FLT_MAX, hi = -FLT_MAX;
        for (int s = 0; s < 8; s++)
            if (used & (1u << s)) { lo = fminf(lo, klo[s][a]); hi = fmaxf(hi, khi[s][a]); }
        if (!(lo <= hi)) { lo = 0.0f; hi = 0.0f; }
        const double extent = (double)hi - (double)lo;
        int e = -100;
        if (extent > 0.0) { int ex; frexp(extent / 376.0, &ex); e = ex; }
        const double amax = fmax(fabs((double)lo), fabs((double)hi));
        if (amax > 0.0) e = max(e, ilogb(amax) - 23);
        e = min(126, max(-100, e));
        const double cell = ldexp(1.0, e);
        const double pd = (double)lo - 128.0 * cell;
        float pf = (float)pd;
        if ((double)pf > pd) pf = nextafterf(pf, -FLT_MAX);
        node.p[a] = pf;
        node.e[a] = (uint8_t)(e + 127);
        uint8_t* qlo = a == 0 ? node.lox : (a == 1 ? node.loy : node.loz);
        uint8_t* qhi = a == 0 ? node.hix : (a == 1 ? node.hiy : node.hiz);
        for (int s = 0; s < 8; s++)
        {
            qlo[s] = 255; qhi[s] = 0;
            if (!(used & (1u << s))) continue;
            long long vl = (long long)floor(((double)klo[s][a] - (double)pf) / cell);
            long long vh = (long long)ceil(((double)khi[s][a] - (double)pf) / cell);
            if (vl < 128 || vh > 510) *overflow = 1;
            vl = min(510LL, max(128LL, vl)); vh = min(510LL, max(128LL, vh));
            if (vl >= 256) vl &= ~1LL;
            if (vh >= 256 && (vh & 1)) vh++;
            if (vh > 510) { *overflow = 1; vh = 510; }
            qlo[s] = (uint8_t)(vl < 256 ? vl - 128 : vl / 2);
            qhi[s] = (uint8_t)(vh < 256 ? vh - 128 : vh / 2);
        }
    }
}

} // namespace b200rt
