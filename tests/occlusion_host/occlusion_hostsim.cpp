// occlusion_hostsim.cpp — TEST-ONLY: compiles the device header csrc/rt_trace.cuh (exact policy) with g++ and drives the
// occlusion kernel's per-ray function on the host, so that it can be checked against the CPU reference
// (tests/rays_host/rays_reference.c) on a machine without a GPU.  It is NOT part of the product and is never loaded by
// the package: only tests/test_occlusion.py loads it.
#define RT_TU_EXACT 1
#include "../../rust-swift-raytracer_b200/csrc/rt_trace.cuh"
#include "../../rust-swift-raytracer_b200/csrc/rt_host.hpp"

#include <cmath>
#include <cstring>

namespace rt {
struct DeviceScene {};
World::World()  = default;
World::~World() = default;
void World::invalidate_device() { packed_.reset(); }
}   // namespace rt

// TEST-ONLY: rt_trace.cuh ray_occluded (which rt_occlusion_kernel calls per lane) for n rays of 8 floats each, one
// byte per ray.  flags: bit 31 selects the FILTER walk, bit 30 the CULL walk (as rays_hostsim), else the direct loops.
// Returns 0 on success.
extern "C" int hostsim_occluded_rays(const char* scene_text, size_t n, const float* rays, uint32_t flags,
                                     uint8_t* occluded)
{
    using namespace rt;
    ParseResult pr = parse_input(scene_text, std::strlen(scene_text));
    if (pr.error != ParseError::Ok) return (int)pr.error;
    const World::Packed& pk = pr.world->packed();
    RtSceneView G = pk.view(pk.blob.data());
    if ((flags & 0x40000000u) && G.n_groups == 0) return 100;      // the world has no block C (< 64 spheres)
    CullView cv{G.cull_bound, G.cull_sph, G.cull_r2, G.cull_orig, G.n_groups};
    for (size_t i = 0; i < n; ++i) {
        RtFloat4 r0, r1;
        std::memcpy(&r0, rays + 8 * i, 16);
        std::memcpy(&r1, rays + 8 * i + 4, 16);
        uint32_t a;
        if (flags & 0x40000000u)      a = ray_occluded<RT_SPH_CULL, true>(G, G.sph_filter, G.sph_r2, cv, G.tri_plane, r0, r1, 1.0f);
        else if (flags & 0x80000000u) a = ray_occluded<RT_SPH_FILTER, true>(G, G.sph_filter, G.sph_r2, cv, G.tri_plane, r0, r1, 1.0f);
        else if (G.n_tri_pad)         a = ray_occluded<RT_SPH_DIRECT, true>(G, G.sph, nullptr, cv, G.tri_plane, r0, r1, 1.0f);
        else                          a = ray_occluded<RT_SPH_DIRECT, false>(G, G.sph, nullptr, cv, G.tri_plane, r0, r1, 1.0f);
        occluded[i] = (uint8_t)a;
    }
    return 0;
}
