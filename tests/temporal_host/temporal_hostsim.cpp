// temporal_hostsim.cpp — TEST-ONLY: compiles temporal accumulation's device header csrc/rt_temporal.cuh with g++ and
// runs its per-pixel functions over a whole frame as rt_temporal.cu runs them (the host's projection set-up, then
// tp_pixel and tp_rgba8 per pixel), so that they can be checked against the numpy reference of tests/test_temporal.py
// on a machine without a GPU.  It is NOT part of the product and is never loaded by the package.
#define RT_TU_EXACT 1
#include "../../rust-swift-raytracer_b200/csrc/rt_temporal.cuh"

#include <cstring>

// accum float4 [H][W], position / normal [H][W][3], prim [H][W], camera 12 floats.  prev_camera NULL: no history (the
// other prev_* are then not read).  max_history, normal_cos, plane_tol: the options after defaults.  pixels may be
// NULL.  The mode rule is rt::temporal's: a previous camera equal bit for bit takes the pixel itself as its one tap.
extern "C" int hostsim_temporal(uint32_t W, uint32_t H, const float* accum, int32_t spp, const float* position,
                                const float* normal, const int32_t* prim, const float* camera, const float* prev_camera,
                                const float* prev_position, const float* prev_normal, const int32_t* prev_prim,
                                const float* prev_color, const float* prev_length, uint32_t max_history,
                                float normal_cos, float plane_tol, float* color, float* length, uint32_t* pixels)
{
    using namespace rt;
    RtTemporalParams P{};
    P.accum         = reinterpret_cast<const RtFloat4*>(accum);
    P.position      = position;
    P.normal        = normal;
    P.prim          = prim;
    P.prev_color    = reinterpret_cast<const RtFloat4*>(prev_color);
    P.prev_length   = prev_length;
    P.prev_position = prev_position;
    P.prev_normal   = prev_normal;
    P.prev_prim     = prev_prim;
    P.width         = W;
    P.height        = H;
    P.mode          = !prev_camera ? RT_TEMPORAL_NO_HISTORY
                      : std::memcmp(camera, prev_camera, 12 * sizeof(float)) == 0 ? RT_TEMPORAL_SAME_CAMERA
                                                                                  : RT_TEMPORAL_REPROJECT;
    P.k             = 1.0f / (float)spp;
    P.spp           = (float)spp;
    P.max_history   = (float)max_history;
    P.normal_cos    = normal_cos;
    P.plane_tol     = plane_tol;
    P.wm1           = (float)(W - 1u);
    P.hm1           = (float)(H - 1u);
    P.fw            = (float)W;
    P.fh            = (float)H;
    if (P.mode == RT_TEMPORAL_REPROJECT) tp_setup_projection(P, prev_camera);
    for (uint32_t y = 0; y < H; ++y)
        for (uint32_t x = 0; x < W; ++x) {
            const size_t p = (size_t)y * W + x;
            RtFloat4     c;
            float        len;
            tp_pixel(P, x, y, c, len);
            color[4 * p] = c.x; color[4 * p + 1] = c.y; color[4 * p + 2] = c.z; color[4 * p + 3] = c.w;
            length[p] = len;
            if (pixels) pixels[p] = tp_rgba8(c);
        }
    return 0;
}
