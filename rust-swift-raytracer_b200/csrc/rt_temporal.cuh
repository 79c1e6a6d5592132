// rt_temporal.cuh — the per-pixel functions of temporal accumulation (rt_temporal.cu), written once for the device and,
// for the CPU tests, compilable as plain C++ (tests/temporal_host).  A pixel's colour history is looked up where its
// surface was in the previous frame (the projection of its first-hit position into the previous camera, bilinear taps
// accepted by normal and plane distance) and blended with the frame's new samples; DESIGN.md §15 is the contract.
//
// Exact arithmetic only: the device TU is compiled with --fmad=false and the host build with -ffp-contract=off, every
// expression below is evaluated left to right as written and divides are IEEE `/`.  The GPU result then equals the CPU
// reference bit for bit.
#pragma once
#include "rt_trace.cuh"     // RT_HD, resolve_pixel

namespace rt {

constexpr float kTemporalMinWeight = 0x1p-7f;   // accepted bilinear weight below this: no history

RT_HD float tp_load(const float* p)
{
#if defined(__CUDA_ARCH__)
    return __ldg(p);
#else
    return *p;
#endif
}

RT_HD int32_t tp_load(const int32_t* p)
{
#if defined(__CUDA_ARCH__)
    return __ldg(p);
#else
    return *p;
#endif
}

RT_HD RtFloat4 tp_load(const RtFloat4* p)
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
RT_HD float tp_dot(float ax, float ay, float az, float bx, float by, float bz)
{
    return (ax * bx + ay * by) + az * bz;
}

// cross(a, b) = (a.y*b.z - a.z*b.y, a.z*b.x - a.x*b.z, a.x*b.y - a.y*b.x)
RT_HD RtVec3 tp_cross(const RtVec3& a, const RtVec3& b)
{
    RtVec3 r;
    r.x = a.y * b.z - a.z * b.y;
    r.y = a.z * b.x - a.x * b.z;
    r.z = a.x * b.y - a.y * b.x;
    return r;
}

RT_HD bool tp_finite(float v) { return fabsf(v) <= 3.40282347e38f; }   // false for +-inf and NaN

// The projection constants of the previous camera (camera12: origin, lower_left_corner, horizontal, vertical), once per
// call on the host.
RT_HD void tp_setup_projection(RtTemporalParams& P, const float prev[12])
{
    const RtVec3 o = {prev[0], prev[1], prev[2]}, h = {prev[6], prev[7], prev[8]}, v = {prev[9], prev[10], prev[11]};
    const RtVec3 a = {prev[3] - o.x, prev[4] - o.y, prev[5] - o.z};
    P.prev_origin = o;
    P.cn          = tp_cross(h, v);
    P.cs          = tp_cross(v, a);
    P.ct          = tp_cross(a, h);
    P.det         = tp_dot(a.x, a.y, a.z, P.cn.x, P.cn.y, P.cn.z);
}

// The continuous previous pixel (x, y) of the surface point X: false when X is not in front of the previous camera or
// (x, y) is NaN or outside [-1, W] x [-1, H].  (u', t') solve w = s ((a + h' u') + v' t') by Cramer's rule, with
// w = X - o' and s = den / det; x, y invert pixel_uv at jitter (0.5, 0.5) and the row flip.
RT_HD bool tp_project(const RtTemporalParams& P, float X0, float X1, float X2, float& x, float& y)
{
    const float wx = X0 - P.prev_origin.x, wy = X1 - P.prev_origin.y, wz = X2 - P.prev_origin.z;
    const float den = tp_dot(wx, wy, wz, P.cn.x, P.cn.y, P.cn.z);
    if (den == 0.0f || (den > 0.0f) != (P.det > 0.0f)) return false;
    const float u = tp_dot(wx, wy, wz, P.cs.x, P.cs.y, P.cs.z) / den;
    const float t = tp_dot(wx, wy, wz, P.ct.x, P.ct.y, P.ct.z) / den;
    x             = u * P.wm1 - 0.5f;
    const float r = t * P.hm1 - 0.5f;
    y             = P.hm1 - r;
    return x >= -1.0f && x <= P.fw && y >= -1.0f && y <= P.fh;
}

struct TpSums {
    float w, r, g, b, a, len;   // accepted weights, and the weighted previous colour and length
};

// Whether tap (qx, qy) of the previous frame with bilinear weight w counts for the hit pixel with normal n and position
// X: it lies inside the frame, is a hit, faces like the pixel (dot(n, n_q) >= normal_cos), lies on its tangent plane
// (|dot(n, X_q - X)| <= plane_tol) and w > 0.  q: its index, set when the tap lies inside the frame.
RT_HD bool tp_accept(const RtTemporalParams& P, int qx, int qy, float w, float nx, float ny, float nz, float X0,
                     float X1, float X2, size_t& q)
{
    if (qx < 0 || qy < 0 || qx >= (int)P.width || qy >= (int)P.height || !(w > 0.0f)) return false;   // W, H < 2^30
    q = (size_t)qy * P.width + (size_t)qx;
    if (tp_load(P.prev_prim + q) < 0) return false;
    const float* nq = P.prev_normal + 3 * q;
    if (!(tp_dot(nx, ny, nz, tp_load(nq), tp_load(nq + 1), tp_load(nq + 2)) >= P.normal_cos)) return false;
    const float* xq = P.prev_position + 3 * q;
    const float  d  = tp_dot(nx, ny, nz, tp_load(xq) - X0, tp_load(xq + 1) - X1, tp_load(xq + 2) - X2);
    return fabsf(d) <= P.plane_tol;
}

// Tap (qx, qy) of the previous frame with bilinear weight w, for the hit pixel with normal n and position X: added to
// s when tp_accept takes it.
RT_HD void tp_tap(const RtTemporalParams& P, int qx, int qy, float w, float nx, float ny, float nz, float X0, float X1,
                  float X2, TpSums& s)
{
    size_t q;
    if (!tp_accept(P, qx, qy, w, nx, ny, nz, X0, X1, X2, q)) return;
    const RtFloat4 c = tp_load(P.prev_color + q);
    s.w   = s.w + w;
    s.r   = s.r + w * c.x;
    s.g   = s.g + w * c.y;
    s.b   = s.b + w * c.z;
    s.a   = s.a + w * c.w;
    s.len = s.len + w * tp_load(P.prev_length + q);
}

// The output of pixel (column, row): the mean m = sum * k with length spp when the pixel has no history, else the
// history (weighted mean of the accepted taps, its length capped at max_history) blended with the new sums.
RT_HD void tp_pixel(const RtTemporalParams& P, uint32_t column, uint32_t row, RtFloat4& color, float& length)
{
    const size_t   p   = (size_t)row * P.width + column;
    const RtFloat4 sum = tp_load(P.accum + p);
    color.x = sum.x * P.k; color.y = sum.y * P.k; color.z = sum.z * P.k; color.w = sum.w * P.k;
    length  = P.spp;
    if (P.mode == RT_TEMPORAL_NO_HISTORY || tp_load(P.prim + p) < 0) return;
    const float X0 = tp_load(P.position + 3 * p), X1 = tp_load(P.position + 3 * p + 1), X2 = tp_load(P.position + 3 * p + 2);
    const float nx = tp_load(P.normal + 3 * p), ny = tp_load(P.normal + 3 * p + 1), nz = tp_load(P.normal + 3 * p + 2);
    if (!(tp_finite(X0) && tp_finite(X1) && tp_finite(X2) && tp_finite(nx) && tp_finite(ny) && tp_finite(nz))) return;
    TpSums s = {0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f};
    if (P.mode == RT_TEMPORAL_SAME_CAMERA) {
        tp_tap(P, (int)column, (int)row, 1.0f, nx, ny, nz, X0, X1, X2, s);
    } else {
        float x, y;
        if (!tp_project(P, X0, X1, X2, x, y)) return;
        const float x0 = floorf(x), y0 = floorf(y);
        const float fx = x - x0, fy = y - y0;
        const int   ix = (int)x0, iy = (int)y0;                                       // in [-1, 2^30]
        tp_tap(P, ix, iy, (1.0f - fx) * (1.0f - fy), nx, ny, nz, X0, X1, X2, s);
        tp_tap(P, ix + 1, iy, fx * (1.0f - fy), nx, ny, nz, X0, X1, X2, s);
        tp_tap(P, ix, iy + 1, (1.0f - fx) * fy, nx, ny, nz, X0, X1, X2, s);
        tp_tap(P, ix + 1, iy + 1, fx * fy, nx, ny, nz, X0, X1, X2, s);
    }
    if (s.w < kTemporalMinWeight) return;
    const float n = fminf(s.len / s.w, P.max_history);
    if (!(n > 0.0f)) return;
    const float L = n + P.spp;
    color.x = ((s.r / s.w) * n + sum.x) / L;
    color.y = ((s.g / s.w) * n + sum.y) / L;
    color.z = ((s.b / s.w) * n + sum.z) / L;
    color.w = ((s.a / s.w) * n + sum.w) / L;
    length  = L;
}

RT_HD uint32_t tp_rgba8(const RtFloat4& c) { return resolve_pixel<false>(c.x, c.y, c.z, c.w, 1); }

}   // namespace rt
