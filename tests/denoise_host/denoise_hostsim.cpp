// denoise_hostsim.cpp — TEST-ONLY: compiles the denoiser's device header csrc/rt_denoise.cuh with g++ and runs its
// per-pixel functions over a whole frame in the order the kernels of rt_denoise.cu run them (pack, iterations, the
// fused last iteration), so that they can be checked against the numpy reference of tests/test_denoise.py on a machine
// without a GPU.  It is NOT part of the product and is never loaded by the package.
#define RT_TU_EXACT 1
#include "../../rust-swift-raytracer_b200/csrc/rt_denoise.cuh"

#include <vector>

// accum float4 [H][W], normal / position / albedo [H][W][3], prim [H][W]; sc, sn, sx: the scales 1/((16 s) s).
// pixels (RGBA8 [H][W]) and color (float4 [H][W]) may each be NULL.  Returns 0.
extern "C" int hostsim_denoise(uint32_t W, uint32_t H, const float* accum, int32_t spp, const float* normal,
                               const float* position, const float* albedo, const int32_t* prim, uint32_t iterations,
                               float sc, float sn, float sx, uint32_t* pixels, float* color)
{
    using namespace rt;
    const size_t          n = (size_t)W * H;
    const RtFloat4*       sums = reinterpret_cast<const RtFloat4*>(accum);
    std::vector<RtFloat4> e0(n), e1(n), gn(n), gx(n);
    RtFloat4*             e[2] = {e0.data(), e1.data()};
    const float           k = 1.0f / (float)spp;
    for (size_t i = 0; i < n; ++i)
        dn_pack_pixel(sums[i], k, albedo[3 * i], albedo[3 * i + 1], albedo[3 * i + 2], normal[3 * i], normal[3 * i + 1],
                      normal[3 * i + 2], position[3 * i], position[3 * i + 1], position[3 * i + 2], prim[i], e0[i],
                      gn[i], gx[i]);
    for (uint32_t it = 0; it < iterations; ++it) {
        const bool  last = it + 1 == iterations;
        const float sc_i = sc * (float)(1u << (2u * it));
        for (uint32_t y = 0; y < H; ++y)
            for (uint32_t x = 0; x < W; ++x) {
                const size_t p    = (size_t)y * W + x;
                const bool   miss = gn[p].w != 0.0f;
                RtFloat4     f{0.f, 0.f, 0.f, 0.f};
                if (!miss) f = dn_filter_pixel(e[it & 1u], gn.data(), gx.data(), W, H, x, y, 1u << it, sc_i, sn, sx);
                if (!last) {
                    if (!miss) e[(it + 1u) & 1u][p] = f;
                    continue;
                }
                const RtFloat4 c = dn_finish_pixel(sums[p], k, albedo[3 * p], albedo[3 * p + 1], albedo[3 * p + 2], miss, f);
                if (color) { color[4 * p] = c.x; color[4 * p + 1] = c.y; color[4 * p + 2] = c.z; color[4 * p + 3] = c.w; }
                if (pixels) pixels[p] = dn_rgba8(c);
            }
    }
    return 0;
}
