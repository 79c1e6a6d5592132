// svgf_hostsim.cpp — TEST-ONLY: compiles variance-guided filtering's device header csrc/rt_svgf.cuh with g++ and runs
// its per-pixel functions over a whole frame as the three kernels of rt_svgf.cu run them (the host's projection set-up,
// then the temporal pass, the variance pass and the a-trous iterations, each over every pixel before the next), so that
// they can be checked against the numpy reference of tests/test_svgf.py on a machine without a GPU.  It is NOT part of
// the product and is never loaded by the package.
#define RT_TU_EXACT 1
#include "../../rust-swift-raytracer_b200/csrc/rt_svgf.cuh"

#include <cstring>
#include <vector>

// accum float4 [H][W], position / normal / albedo [H][W][3], prim [H][W], camera 12 floats.  prev_camera NULL: no
// history (the other prev_* are then not read).  The options after defaults; sigma_* are the sigmas themselves.  The
// outputs illum float4, moments float2, length, color float4 and pixels RGBA8 are all written.  The mode rule is
// rt::svgf's: a previous camera equal bit for bit takes the pixel itself as its one tap.
extern "C" int hostsim_svgf(uint32_t W, uint32_t H, const float* accum, int32_t spp, const float* position,
                            const float* normal, const float* albedo, const int32_t* prim, const float* camera,
                            const float* prev_camera, const float* prev_position, const float* prev_normal,
                            const int32_t* prev_prim, const float* prev_illum, const float* prev_moments,
                            const float* prev_length, uint32_t iterations, uint32_t max_history, float normal_cos,
                            float plane_tol, float sigma_luminance, float sigma_normal, float sigma_plane, float* illum,
                            float* moments, float* length, float* color, uint32_t* pixels)
{
    using namespace rt;
    const size_t n = (size_t)W * H;
    std::vector<RtFloat4> e0(n), e1(n), gn(n), gx(n);
    std::vector<float>    v0(n), v1(n);
    RtSvgfParams P{};
    RtTemporalParams& T = P.t;
    T.accum         = reinterpret_cast<const RtFloat4*>(accum);
    T.position      = position;
    T.normal        = normal;
    T.prim          = prim;
    T.prev_color    = reinterpret_cast<const RtFloat4*>(prev_illum);
    T.prev_length   = prev_length;
    T.prev_position = prev_position;
    T.prev_normal   = prev_normal;
    T.prev_prim     = prev_prim;
    T.width         = W;
    T.height        = H;
    T.mode          = !prev_camera ? RT_TEMPORAL_NO_HISTORY
                      : std::memcmp(camera, prev_camera, 12 * sizeof(float)) == 0 ? RT_TEMPORAL_SAME_CAMERA
                                                                                  : RT_TEMPORAL_REPROJECT;
    T.k             = 1.0f / (float)spp;
    T.spp           = (float)spp;
    T.max_history   = (float)max_history;
    T.normal_cos    = normal_cos;
    T.plane_tol     = plane_tol;
    T.wm1           = (float)(W - 1u);
    T.hm1           = (float)(H - 1u);
    T.fw            = (float)W;
    T.fh            = (float)H;
    if (T.mode == RT_TEMPORAL_REPROJECT) tp_setup_projection(T, prev_camera);
    P.albedo       = albedo;
    P.prev_moments = reinterpret_cast<const RtFloat2*>(prev_moments);
    P.illum        = reinterpret_cast<RtFloat4*>(illum);
    P.moments      = reinterpret_cast<RtFloat2*>(moments);
    P.length       = length;
    P.color        = reinterpret_cast<RtFloat4*>(color);
    P.pixels       = pixels;
    P.e[0] = e0.data(); P.e[1] = e1.data(); P.var[0] = v0.data(); P.var[1] = v1.data();
    P.gn = gn.data(); P.gx = gx.data();
    P.iterations = iterations;
    P.spp4       = 4.0f * (float)spp;
    P.ql         = (16.0f * sigma_luminance) * sigma_luminance;
    P.sn         = dn_scale(sigma_normal);
    P.sx         = dn_scale(sigma_plane);
    for (uint32_t y = 0; y < H; ++y)                                         // rt_svgf_temporal_kernel
        for (uint32_t x = 0; x < W; ++x) {
            const size_t p = (size_t)y * W + x;
            sv_temporal_pixel(P, x, y, P.e[0][p], P.moments[p], P.length[p], P.gn[p], P.gx[p]);
        }
    for (uint32_t y = 0; y < H; ++y)                                         // rt_svgf_variance_kernel
        for (uint32_t x = 0; x < W; ++x) {
            const size_t p = (size_t)y * W + x;
            if (P.gn[p].w == 0.0f) P.var[0][p] = sv_variance_pixel(P, P.moments, P.length, x, y);
        }
    for (uint32_t it = 0; it < iterations; ++it) {                           // rt_svgf_iter_kernel<FIRST, LAST>
        const bool first = it == 0, last = it + 1 == iterations;
        for (uint32_t y = 0; y < H; ++y)
            for (uint32_t x = 0; x < W; ++x) {
                const size_t p    = (size_t)y * W + x;
                const bool   miss = P.gn[p].w != 0.0f;
                RtFloat4     f    = {0.0f, 0.0f, 0.0f, 0.0f};
                float        var  = 0.0f;
                if (!miss) f = sv_filter_pixel(P, P.e[it & 1u], P.var[it & 1u], x, y, 1u << it, var);
                if (first) P.illum[p] = miss ? P.e[0][p] : f;
                if (!last) {
                    if (!miss) { P.e[(it + 1u) & 1u][p] = f; P.var[(it + 1u) & 1u][p] = var; }
                    continue;
                }
                const float*   a = albedo + 3 * p;
                const RtFloat4 c = dn_finish_pixel(T.accum[p], T.k, a[0], a[1], a[2], miss, f);
                P.color[p]  = c;
                P.pixels[p] = dn_rgba8(c);
            }
    }
    return 0;
}
