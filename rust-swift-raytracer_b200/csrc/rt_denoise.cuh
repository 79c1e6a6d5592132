// rt_denoise.cuh — the per-pixel functions of the denoiser (rt_denoise.cu), written once for the device and, for the
// CPU tests, compilable as plain C++ (tests/denoise_host).  Edge-avoiding a-trous wavelet filter (Dammertz et al.,
// HPG 2010) of the demodulated colour, guided by the first-hit normal and position; DESIGN.md §12 is the contract.
//
// Exact arithmetic only: the device TU is compiled with --fmad=false and the host build with -ffp-contract=off, every
// expression below is evaluated left to right as written, divides are IEEE `/`, and nothing calls expf (the device
// library and glibc differ there).  The GPU result then equals the CPU reference bit for bit.
#pragma once
#include "rt_trace.cuh"     // RT_HD, resolve_pixel

namespace rt {

constexpr float kDenoiseAlbedoFloor = 0x1p-10f;   // a' = max(albedo, 2^-10) per channel

// B3-spline taps h[-2..2]
RT_HD float dn_tap(int d)
{
    return d == 0 ? 0.375f : (d == 1 || d == -1) ? 0.25f : 0.0625f;
}

RT_HD RtFloat4 dn_load(const RtFloat4* p)
{
#if defined(__CUDA_ARCH__)
    const float4 v = __ldg(reinterpret_cast<const float4*>(p));
    RtFloat4     r;
    r.x = v.x; r.y = v.y; r.z = v.z; r.w = v.w;
    return r;
#else
    return *p;
#endif
}

// dot(a, b) = (a.x*b.x + a.y*b.y) + a.z*b.z
RT_HD float dn_dot(float ax, float ay, float az, float bx, float by, float bz)
{
    return (ax * bx + ay * by) + az * bz;
}

// Demodulation of one pixel: the mean m = sum * k; e = m / a' (rgb) on a hit.  gn = (normal, 1 on a miss else 0),
// gx = (position, 0).
RT_HD void dn_pack_pixel(RtFloat4 sum, float k, float ax, float ay, float az, float nx, float ny, float nz, float px,
                         float py, float pz, int32_t prim, RtFloat4& e, RtFloat4& gn, RtFloat4& gx)
{
    const float mx = sum.x * k, my = sum.y * k, mz = sum.z * k;
    e.x = mx / fmaxf(ax, kDenoiseAlbedoFloor);
    e.y = my / fmaxf(ay, kDenoiseAlbedoFloor);
    e.z = mz / fmaxf(az, kDenoiseAlbedoFloor);
    e.w = 0.0f;
    gn.x = nx; gn.y = ny; gn.z = nz; gn.w = prim < 0 ? 1.0f : 0.0f;
    gx.x = px; gx.y = py; gx.z = pz; gx.w = 0.0f;
}

// Weight of tap q for pixel p: hxy * r^16 with r = 1 / ((1 + u_c) (1 + u_n) (1 + u_x)), (1 + u/16)^-16 ~ exp(-u).
RT_HD float dn_weight(float hxy, const RtFloat4& ep, const RtFloat4& np, const RtFloat4& xp, const RtFloat4& eq,
                      const RtFloat4& nq, const RtFloat4& xq, float sc_i, float sn, float sx)
{
    const float cx = ep.x - eq.x, cy = ep.y - eq.y, cz = ep.z - eq.z;
    const float uc = dn_dot(cx, cy, cz, cx, cy, cz) * sc_i;
    const float nx = np.x - nq.x, ny = np.y - nq.y, nz = np.z - nq.z;
    const float un = dn_dot(nx, ny, nz, nx, ny, nz) * sn;
    const float d  = dn_dot(np.x, np.y, np.z, xq.x - xp.x, xq.y - xp.y, xq.z - xp.z);
    const float ux = (d * d) * sx;
    float r = 1.0f / (((1.0f + uc) * (1.0f + un)) * (1.0f + ux));
    r = r * r;
    r = r * r;
    r = r * r;
    r = r * r;
    return hxy * r;
}

// One a-trous iteration at hit pixel (x, y) with step s: the weighted mean of the accepted taps, in the order dy = -2..2
// (outer), dx = -2..2 (inner).  A tap outside the frame, at a miss pixel, or whose weight is not > 0 is skipped; if none
// is accepted the pixel keeps its value.  e, gn, gx: the packed frame (dn_pack_pixel).
RT_HD RtFloat4 dn_filter_pixel(const RtFloat4* e, const RtFloat4* gn, const RtFloat4* gx, uint32_t width,
                               uint32_t height, uint32_t x, uint32_t y, uint32_t s, float sc_i, float sn, float sx)
{
    const size_t   p  = (size_t)y * width + x;
    const RtFloat4 ep = dn_load(e + p), np = dn_load(gn + p), xp = dn_load(gx + p);
    float sw = 0.0f, sr = 0.0f, sg = 0.0f, sb = 0.0f;
#pragma unroll
    for (int dy = -2; dy <= 2; ++dy) {
        const int qy = (int)y + dy * (int)s;                                  // |x|, |y| < 2^30, s <= 512
        if (qy < 0 || qy >= (int)height) continue;
#pragma unroll
        for (int dx = -2; dx <= 2; ++dx) {
            const int qx = (int)x + dx * (int)s;
            if (qx < 0 || qx >= (int)width) continue;
            const size_t   q  = (size_t)qy * width + (size_t)qx;
            const RtFloat4 nq = dn_load(gn + q);
            if (nq.w != 0.0f) continue;                                        // a miss is never a neighbour
            const RtFloat4 eq = dn_load(e + q), xq = dn_load(gx + q);
            const float    w  = dn_weight(dn_tap(dx) * dn_tap(dy), ep, np, xp, eq, nq, xq, sc_i, sn, sx);
            if (!(w > 0.0f)) continue;                                         // also NaN
            sw = sw + w;
            sr = sr + w * eq.x;
            sg = sg + w * eq.y;
            sb = sb + w * eq.z;
        }
    }
    if (!(sw > 0.0f)) return ep;
    RtFloat4 r;
    r.x = sr / sw; r.y = sg / sw; r.z = sb / sw; r.w = 0.0f;
    return r;
}

// The output of one pixel: a hit gives (f * a', m.a), a miss its mean m; RGBA8 = resolve_pixel of that colour with
// spp 1 (so a miss pixel's RGBA8 is the render's own RGBA8 of the same sums).
RT_HD RtFloat4 dn_finish_pixel(RtFloat4 sum, float k, float ax, float ay, float az, bool miss, const RtFloat4& f)
{
    RtFloat4 c;
    c.x = sum.x * k; c.y = sum.y * k; c.z = sum.z * k; c.w = sum.w * k;
    if (!miss) {
        c.x = f.x * fmaxf(ax, kDenoiseAlbedoFloor);
        c.y = f.y * fmaxf(ay, kDenoiseAlbedoFloor);
        c.z = f.z * fmaxf(az, kDenoiseAlbedoFloor);
    }
    return c;
}

RT_HD uint32_t dn_rgba8(const RtFloat4& c) { return resolve_pixel<false>(c.x, c.y, c.z, c.w, 1); }

// sigma -> 1 / ((16 sigma) sigma), in float32 (the host computes the three scales once per call)
RT_HD float dn_scale(float sigma) { return 1.0f / ((16.0f * sigma) * sigma); }

}   // namespace rt
