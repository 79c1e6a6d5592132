// rt_svgf.cuh — the per-pixel functions of variance-guided filtering (rt_svgf.cu), written once for the device and, for
// the CPU tests, compilable as plain C++ (tests/svgf_host).  SVGF (Schied et al., HPG 2017) joins temporal accumulation
// (§15) and the a-trous filter (§12): the first two luminance moments travel with the reprojected colour history, give
// each pixel a variance estimate, and that variance sets the pixel's colour weight in the filter.  DESIGN.md §16 is the
// contract.
//
// Exact arithmetic only: the device TU is compiled with --fmad=false and the host build with -ffp-contract=off, every
// expression below is evaluated left to right as written, divides are IEEE `/`, and nothing calls expf or sqrtf.  The
// GPU result then equals the CPU reference bit for bit.
#pragma once
#include "rt_temporal.cuh"   // tp_load, tp_finite, tp_project, tp_accept
#include "rt_denoise.cuh"    // dn_pack_pixel, dn_weight, dn_tap, dn_finish_pixel

namespace rt {

constexpr float kSvgfEps = 0x1p-20f;   // il = 1 / (ql * g + eps): a pixel of variance 0 still tolerates 2^-20 of lum^2

RT_HD RtFloat2 sv_load(const RtFloat2* p)
{
#if defined(__CUDA_ARCH__)
    const float2 v = __ldg(reinterpret_cast<const float2*>(p));
    RtFloat2     r;
    r.x = v.x; r.y = v.y;
    return r;
#else
    return *p;
#endif
}

// lum(e) = (0.2126 r + 0.7152 g) + 0.0722 b
RT_HD float sv_lum(float r, float g, float b) { return (0.2126f * r + 0.7152f * g) + 0.0722f * b; }

struct SvSums {
    float w, r, g, b, m1, m2, len;   // accepted weights, and the weighted previous illum, moments and length
};

// Tap (qx, qy) of the previous frame: added to s when tp_accept takes it (§15.1's rule, unchanged).
RT_HD void sv_tap(const RtSvgfParams& P, int qx, int qy, float w, float nx, float ny, float nz, float X0, float X1,
                  float X2, SvSums& s)
{
    size_t q;
    if (!tp_accept(P.t, qx, qy, w, nx, ny, nz, X0, X1, X2, q)) return;
    const RtFloat4 c = tp_load(P.t.prev_color + q);
    const RtFloat2 m = sv_load(P.prev_moments + q);
    s.w   = s.w + w;
    s.r   = s.r + w * c.x;
    s.g   = s.g + w * c.y;
    s.b   = s.b + w * c.z;
    s.m1  = s.m1 + w * m.x;
    s.m2  = s.m2 + w * m.y;
    s.len = s.len + w * tp_load(P.t.prev_length + q);
}

// Stage 1 at pixel (column, row): the demodulated colour e and its luminance moments (l, l*l), blended with the
// history found as §15 finds it.  illum: (rgb, lum(rgb)) at a hit, m at a miss; gn, gx: the packed guides.
RT_HD void sv_temporal_pixel(const RtSvgfParams& P, uint32_t column, uint32_t row, RtFloat4& illum, RtFloat2& moments,
                             float& length, RtFloat4& gn, RtFloat4& gx)
{
    const RtTemporalParams& T = P.t;
    const size_t   p   = (size_t)row * T.width + column;
    const RtFloat4 sum = tp_load(T.accum + p);
    const int32_t  prim = tp_load(T.prim + p);
    const float X0 = tp_load(T.position + 3 * p), X1 = tp_load(T.position + 3 * p + 1), X2 = tp_load(T.position + 3 * p + 2);
    const float nx = tp_load(T.normal + 3 * p), ny = tp_load(T.normal + 3 * p + 1), nz = tp_load(T.normal + 3 * p + 2);
    const float ax = tp_load(P.albedo + 3 * p), ay = tp_load(P.albedo + 3 * p + 1), az = tp_load(P.albedo + 3 * p + 2);
    RtFloat4 e;
    dn_pack_pixel(sum, T.k, ax, ay, az, nx, ny, nz, X0, X1, X2, prim, e, gn, gx);
    length = T.spp;
    if (prim < 0) {                                                          // a miss: m, no moments
        illum.x = sum.x * T.k; illum.y = sum.y * T.k; illum.z = sum.z * T.k; illum.w = sum.w * T.k;
        moments.x = 0.0f; moments.y = 0.0f;
        return;
    }
    const float l  = sv_lum(e.x, e.y, e.z);
    const float l2 = l * l;
    illum.x = e.x; illum.y = e.y; illum.z = e.z; illum.w = l;
    moments.x = l; moments.y = l2;
    if (T.mode == RT_TEMPORAL_NO_HISTORY) return;
    if (!(tp_finite(X0) && tp_finite(X1) && tp_finite(X2) && tp_finite(nx) && tp_finite(ny) && tp_finite(nz))) return;
    SvSums s = {0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f};
    if (T.mode == RT_TEMPORAL_SAME_CAMERA) {
        sv_tap(P, (int)column, (int)row, 1.0f, nx, ny, nz, X0, X1, X2, s);
    } else {
        float x, y;
        if (!tp_project(T, X0, X1, X2, x, y)) return;
        const float x0 = floorf(x), y0 = floorf(y);
        const float fx = x - x0, fy = y - y0;
        const int   ix = (int)x0, iy = (int)y0;                                       // in [-1, 2^30]
        sv_tap(P, ix, iy, (1.0f - fx) * (1.0f - fy), nx, ny, nz, X0, X1, X2, s);
        sv_tap(P, ix + 1, iy, fx * (1.0f - fy), nx, ny, nz, X0, X1, X2, s);
        sv_tap(P, ix, iy + 1, (1.0f - fx) * fy, nx, ny, nz, X0, X1, X2, s);
        sv_tap(P, ix + 1, iy + 1, fx * fy, nx, ny, nz, X0, X1, X2, s);
    }
    if (s.w < kTemporalMinWeight) return;
    const float n = fminf(s.len / s.w, T.max_history);
    if (!(n > 0.0f)) return;
    const float L = n + T.spp;
    illum.x   = ((s.r / s.w) * n + e.x * T.spp) / L;
    illum.y   = ((s.g / s.w) * n + e.y * T.spp) / L;
    illum.z   = ((s.b / s.w) * n + e.z * T.spp) / L;
    illum.w   = sv_lum(illum.x, illum.y, illum.z);
    moments.x = ((s.m1 / s.w) * n + l * T.spp) / L;
    moments.y = ((s.m2 / s.w) * n + l2 * T.spp) / L;
    length    = L;
}

// The geometric weight r^16, r = 1 / ((1 + u_n) (1 + u_x)), of tap q for pixel p: dn_weight with no colour term.
RT_HD float sv_geometry_weight(const RtFloat4& np, const RtFloat4& xp, const RtFloat4& nq, const RtFloat4& xq, float sn,
                               float sx)
{
    const RtFloat4 zero = {0.0f, 0.0f, 0.0f, 0.0f};
    return dn_weight(1.0f, zero, np, xp, zero, nq, xq, 0.0f, sn, sx);
}

// Stage 2 at hit pixel (x, y): the luminance variance.  From the pixel's own moments once its history holds four
// frames' worth of samples (L >= 4 spp); before that from the moments of the 7x7 neighbourhood (dy = -3..3 outer, dx
// inner; a tap inside the frame and on a hit, weight r^16 > 0), scaled by 4 spp / L.  m, len: stage 1's outputs.
RT_HD float sv_variance_pixel(const RtSvgfParams& P, const RtFloat2* m, const float* len, uint32_t x, uint32_t y)
{
    const uint32_t W = P.t.width, H = P.t.height;
    const size_t   p  = (size_t)y * W + x;
    const float    L  = tp_load(len + p);
    const RtFloat2 mp = sv_load(m + p);
    if (!(L >= P.spp4)) {
        const RtFloat4 np = dn_load(P.gn + p), xp = dn_load(P.gx + p);
        float sw = 0.0f, s1 = 0.0f, s2 = 0.0f;
        for (int dy = -3; dy <= 3; ++dy) {
            const int qy = (int)y + dy;
            if (qy < 0 || qy >= (int)H) continue;
            for (int dx = -3; dx <= 3; ++dx) {
                const int qx = (int)x + dx;
                if (qx < 0 || qx >= (int)W) continue;
                const size_t   q  = (size_t)qy * W + (size_t)qx;
                const RtFloat4 nq = dn_load(P.gn + q);
                if (nq.w != 0.0f) continue;                                    // a miss is never a neighbour
                const float w = sv_geometry_weight(np, xp, nq, dn_load(P.gx + q), P.sn, P.sx);
                if (!(w > 0.0f)) continue;                                     // also NaN
                const RtFloat2 mq = sv_load(m + q);
                sw = sw + w;
                s1 = s1 + w * mq.x;
                s2 = s2 + w * mq.y;
            }
        }
        if (sw > 0.0f) {
            const float mu1 = s1 / sw;
            return fmaxf(s2 / sw - mu1 * mu1, 0.0f) * (P.spp4 / L);
        }
    }
    return fmaxf(mp.y - mp.x * mp.x, 0.0f);
}

// The 3x3 Gaussian {1/4, 1/2, 1/4}^2 of the variance v around hit pixel (x, y), over the taps inside the frame and on
// hits, normalised by their weight.
RT_HD float sv_gauss_variance(const RtSvgfParams& P, const float* v, uint32_t x, uint32_t y)
{
    const uint32_t W = P.t.width, H = P.t.height;
    float sk = 0.0f, sv = 0.0f;
#pragma unroll
    for (int dy = -1; dy <= 1; ++dy) {
        const int qy = (int)y + dy;
        if (qy < 0 || qy >= (int)H) continue;
#pragma unroll
        for (int dx = -1; dx <= 1; ++dx) {
            const int qx = (int)x + dx;
            if (qx < 0 || qx >= (int)W) continue;
            const size_t q = (size_t)qy * W + (size_t)qx;
            if (dn_load(P.gn + q).w != 0.0f) continue;
            const float k = (dx == 0 ? 0.5f : 0.25f) * (dy == 0 ? 0.5f : 0.25f);
            sk = sk + k;
            sv = sv + k * tp_load(v + q);
        }
    }
    return sv / sk;
}

// Stage 3, one a-trous iteration at hit pixel (x, y) with step s: the taps of dn_filter_pixel, each weighted
// h(dx) h(dy) r^16 with r = 1 / ((1 + u_l) (1 + u_n) (1 + u_x)) and u_l = (l_p - l_q)^2 / (ql g + eps), g the 3x3
// Gaussian of the pixel's variance.  Returns the weighted mean colour (luminance in w) and sets var to the variance of
// that mean, sum(w^2 var_q) / (sum w)^2; with no tap accepted the pixel keeps both.
RT_HD RtFloat4 sv_filter_pixel(const RtSvgfParams& P, const RtFloat4* e, const float* v, uint32_t x, uint32_t y,
                               uint32_t s, float& var)
{
    const uint32_t W = P.t.width, H = P.t.height;
    const size_t   p  = (size_t)y * W + x;
    const RtFloat4 ep = dn_load(e + p), np = dn_load(P.gn + p), xp = dn_load(P.gx + p);
    const float    il = 1.0f / (P.ql * sv_gauss_variance(P, v, x, y) + kSvgfEps);
    const RtFloat4 lp = {ep.w, 0.0f, 0.0f, 0.0f};
    float sw = 0.0f, sr = 0.0f, sg = 0.0f, sb = 0.0f, sv = 0.0f;
#pragma unroll
    for (int dy = -2; dy <= 2; ++dy) {
        const int qy = (int)y + dy * (int)s;                                  // |x|, |y| < 2^30, s <= 512
        if (qy < 0 || qy >= (int)H) continue;
#pragma unroll
        for (int dx = -2; dx <= 2; ++dx) {
            const int qx = (int)x + dx * (int)s;
            if (qx < 0 || qx >= (int)W) continue;
            const size_t   q  = (size_t)qy * W + (size_t)qx;
            const RtFloat4 nq = dn_load(P.gn + q);
            if (nq.w != 0.0f) continue;                                        // a miss is never a neighbour
            const RtFloat4 eq = dn_load(e + q), xq = dn_load(P.gx + q);
            const RtFloat4 lq = {eq.w, 0.0f, 0.0f, 0.0f};
            const float    w  = dn_weight(dn_tap(dx) * dn_tap(dy), lp, np, xp, lq, nq, xq, il, P.sn, P.sx);
            if (!(w > 0.0f)) continue;                                         // also NaN
            sw = sw + w;
            sr = sr + w * eq.x;
            sg = sg + w * eq.y;
            sb = sb + w * eq.z;
            sv = sv + (w * w) * tp_load(v + q);
        }
    }
    if (!(sw > 0.0f)) {
        var = tp_load(v + p);
        return ep;
    }
    RtFloat4 r;
    r.x = sr / sw; r.y = sg / sw; r.z = sb / sw; r.w = sv_lum(r.x, r.y, r.z);
    var = sv / (sw * sw);
    return r;
}

}   // namespace rt
