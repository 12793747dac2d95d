// Output stage: an edge-avoiding a-trous wavelet filter standing in for the reference's OIDN "RT" pass
// (Utils::OIDN_denoise, source/utils.cpp:144-196; called three times from main.cpp:118-120 on the tone-mapped frame).
//
// The reference hands the beauty image alone (no albedo / normal guides) to a neural denoiser whose binaries and weights it does
// not ship (.gitignore:14-16), so there is nothing to be bit-compatible with; what is reproduced is the STAGE: RGB in, RGB out,
// same call site (the 13 OIDN C entry points are implemented over this kernel in host/dropin/b200rt_oidn.c), so that the
// reference's unmodified main.cpp writes denoised PNGs that are in fact denoised. Algorithm (Dammertz et al., "Edge-avoiding
// a-trous wavelet transform for fast global illumination filtering", HPG 2010): 5 passes of the 5x5 B3-spline kernel with holes of
// 1, 2, 4, 8, 16 pixels; a tap's weight is the spline weight times exp(-|c_p - c_q|^2 / sigma_i^2) with sigma_i = sigma * 2^-i,
// where c are the pass's input colours; the first pass additionally divides the colour distance by the local luminance deviation
// (3x3), so that noisy flat regions are smoothed and clean edges are not. As in the paper, the weight can also be stopped by
// feature buffers: OIDN's optional "albedo" and "normal" auxiliary images (b200rt_render_aovs computes them), see k_atrous below.
// Without them the filter is colour-guided only, exactly as before guides existed. One thread per pixel; the image (and the
// guides) are a few tens of MB and stay in L2 between passes.
//
// Non-finite pixels are missing data: a pixel with a NaN or +-Inf in R, G or B (a path tracer's NaN, an overflow) gives no tap, is
// left out of the pass-0 luminance statistic, and as the centre is filtered without the colour term (spline times guides over its
// finite taps). A pixel none of whose taps is finite stays non-finite and a wider later pass fills it. Without this, one NaN
// spreads through every weight it touches: 2 * (1 + 2 + 4 + 8 + 16) = 62 pixels in each direction over 5 passes. Alpha is not
// looked at. For finite inputs the arithmetic is unchanged, so is every output bit.
#include <algorithm>

#include "kernels.h"

namespace b200rt {

__device__ __forceinline__ float3 load_rgb(const float* __restrict__ img, int channels, int w, int h, int x, int y)
{
    x = min(max(x, 0), w - 1); y = min(max(y, 0), h - 1);
    const float* p = img + ((size_t)y * w + x) * channels;
    return make_float3(p[0], p[1], p[2]);
}

// Guides (OIDN's auxiliary images, 3 floats per pixel each; a missing one weighs 1): a tap's weight is further multiplied by
// max(0, n_p . n_q)^kSigmaNormal of the normalised guide normals (a zero normal, a miss, matches only zero normals: sky filters
// with sky, geometry does not bleed into it) and by exp(-|a_p - a_q|^2 / kSigmaAlbedo^2). The guides carry the geometric and
// material edges, so the colour term may be more tolerant: its sigma is multiplied by kGuidedColourRelax.
constexpr float kSigmaNormal = 128.0f;
constexpr float kSigmaAlbedo = 0.1f;
constexpr float kGuidedColourRelax = 2.0f;

__device__ __forceinline__ bool finite_rgb(float3 c) { return isfinite(c.x) && isfinite(c.y) && isfinite(c.z); }

// A normal whose float32 squared length is 0 is a miss and comes back as exactly 0. That includes normals too short to square
// (components below ~1e-23): returned as they are, they would pass the zero test below as geometry, match nothing, not even
// themselves, and leave the pixel at 0 / 0.
__device__ __forceinline__ float3 unit_or_zero(float3 n)
{
    const float l2 = n.x * n.x + n.y * n.y + n.z * n.z;
    if (l2 == 0.0f) return make_float3(0.0f, 0.0f, 0.0f);
    const float k = rsqrtf(l2);
    return make_float3(n.x * k, n.y * k, n.z * k);
}

// The colour-only instantiation computes the filter as it was before guides existed, bit for bit on finite images; the guides are
// trailing parameters so that its parameter layout does not move either.
template <bool GUIDED>
__global__ void __launch_bounds__(256) k_atrous(const float* __restrict__ in, int channels, int w, int h, int step, float inv_sigma2, int use_local_noise,
                                                float* __restrict__ out, const float* __restrict__ albedo, const float* __restrict__ normal)
{
    const int x = blockIdx.x * 32 + (threadIdx.x & 31);
    const int y = blockIdx.y * 8 + (threadIdx.x >> 5);
    if (x >= w || y >= h) return;
    const float kern[5] = { 1.0f / 16.0f, 1.0f / 4.0f, 3.0f / 8.0f, 1.0f / 4.0f, 1.0f / 16.0f };
    const float3 c = load_rgb(in, channels, w, h, x, y);
    float3 ca = make_float3(0.0f, 0.0f, 0.0f), cn = ca;
    if constexpr (GUIDED)
    {
        if (albedo) ca = load_rgb(albedo, 3, w, h, x, y);
        if (normal) cn = unit_or_zero(load_rgb(normal, 3, w, h, x, y));
    }
    float noise_scale = 1.0f;
    if (use_local_noise)
    {
        // luminance deviation of the finite pixels of the 3x3 neighbourhood: colour distances are measured in units of it
        float s = 0.0f, s2 = 0.0f, n = 0.0f;
        for (int dy = -1; dy <= 1; dy++)
            for (int dx = -1; dx <= 1; dx++)
            {
                const float3 q = load_rgb(in, channels, w, h, x + dx, y + dy);
                if (!finite_rgb(q)) continue;
                const float l = 0.2126f * q.x + 0.7152f * q.y + 0.0722f * q.z;
                s += l; s2 += l * l; n += 1.0f;
            }
        if (n > 0.0f)
        {
            const float var = fmaxf(s2 / n - (s / n) * (s / n), 0.0f);
            noise_scale = 1.0f / (1.0f + 16.0f * var);      // high local variance -> tolerant weights
        }
    }
    const bool c_finite = finite_rgb(c);
    float3 acc = make_float3(0.0f, 0.0f, 0.0f);
    float wsum = 0.0f;
    for (int j = 0; j < 5; j++)
        for (int i = 0; i < 5; i++)
        {
            const int qx = x + (i - 2) * step, qy = y + (j - 2) * step;
            const float3 q = load_rgb(in, channels, w, h, qx, qy);
            if (!finite_rgb(q)) continue;                   // a missing tap weighs 0
            float wgt = kern[i] * kern[j];
            if (c_finite)
            {
                const float dr = q.x - c.x, dg = q.y - c.y, db = q.z - c.z;
                const float d2 = dr * dr + dg * dg + db * db;
                wgt *= __expf(-d2 * inv_sigma2 * noise_scale);
            }
            if constexpr (GUIDED)
            {
                if (albedo)
                {
                    const float3 a = load_rgb(albedo, 3, w, h, qx, qy);
                    const float ar = a.x - ca.x, ag = a.y - ca.y, ab = a.z - ca.z;
                    wgt *= __expf(-(ar * ar + ag * ag + ab * ab) * (1.0f / (kSigmaAlbedo * kSigmaAlbedo)));
                }
                if (normal)
                {
                    const float3 n = unit_or_zero(load_rgb(normal, 3, w, h, qx, qy));
                    const bool n_zero = n.x == 0.0f && n.y == 0.0f && n.z == 0.0f;
                    const bool c_zero = cn.x == 0.0f && cn.y == 0.0f && cn.z == 0.0f;
                    if (n_zero || c_zero) wgt = n_zero == c_zero ? wgt : 0.0f;
                    else wgt *= __powf(fmaxf(0.0f, n.x * cn.x + n.y * cn.y + n.z * cn.z), kSigmaNormal);
                }
            }
            acc.x += wgt * q.x; acc.y += wgt * q.y; acc.z += wgt * q.z;
            wsum += wgt;
        }
    float* o = out + ((size_t)y * w + x) * channels;
    o[0] = acc.x / wsum; o[1] = acc.y / wsum; o[2] = acc.z / wsum;
    if (channels == 4) o[3] = in[((size_t)y * w + x) * 4 + 3];
}

// blend = blend_factor * denoised + (1 - blend_factor) * noisy (utils.cpp:184-186); alpha -> 1 when present. A missing (non-finite)
// noisy pixel takes the denoised value alone, whatever the blend: 0 * NaN would be NaN.
__global__ void __launch_bounds__(256) k_denoise_blend(const float* __restrict__ noisy, const float* __restrict__ den, int channels, size_t n_px, float blend,
                                                       float* __restrict__ out)
{
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_px; i += (size_t)gridDim.x * blockDim.x)
    {
        const float* p = noisy + i * channels;
        const bool missing = !finite_rgb(make_float3(p[0], p[1], p[2]));
        for (int c = 0; c < 3; c++) out[i * channels + c] = missing ? den[i * channels + c] : blend * den[i * channels + c] + (1.0f - blend) * p[c];
        if (channels == 4) out[i * 4 + 3] = 1.0f;
    }
}

// d_in -> d_out (both w*h*channels floats on the device); d_tmp: scratch of the same size. d_out may alias neither.
cudaError_t launch_denoise(const float* d_in, int channels, const float* d_albedo, const float* d_normal, int w, int h, int iterations,
                           float sigma, float blend, float* d_tmp, float* d_out, cudaStream_t stream)
{
    if (w <= 0 || h <= 0) return cudaSuccess;
    dim3 grid((w + 31) / 32, (h + 7) / 8);
    const float* src = d_in;
    float* bufs[2] = { d_tmp, d_out };
    // arrange the ping-pong so that the last pass lands in d_tmp (the blend then writes d_out)
    int which = (iterations & 1) ? 0 : 1;
    for (int i = 0; i < iterations; i++)
    {
        const float s = sigma / (float)(1 << i);
        float* dst = bufs[which];
        if (d_albedo || d_normal)
        {
            const float sg = s * kGuidedColourRelax;
            k_atrous<true><<<grid, 256, 0, stream>>>(src, channels, w, h, 1 << i, 1.0f / (sg * sg), i == 0 ? 1 : 0, dst, d_albedo, d_normal);
        }
        else k_atrous<false><<<grid, 256, 0, stream>>>(src, channels, w, h, 1 << i, 1.0f / (s * s), i == 0 ? 1 : 0, dst, nullptr, nullptr);
        src = dst;
        which ^= 1;
    }
    const size_t n_px = (size_t)w * h;
    k_denoise_blend<<<(unsigned int)std::min<size_t>((n_px + 255) / 256, 148 * 8), 256, 0, stream>>>(d_in, iterations > 0 ? src : d_in, channels, n_px, blend, d_out);
    return cudaGetLastError();
}

} // namespace b200rt
