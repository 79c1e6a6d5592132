// rays_hostsim.cpp — TEST-ONLY: compiles the device header csrc/rt_trace.cuh (exact policy) with g++ and drives the
// ray-query kernel's per-ray function on the host, so that it can be checked against the CPU reference
// (rays_reference.c) on a machine without a GPU.  It is NOT part of the product and is never loaded by the package:
// only tests/test_rays.py loads it.
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

// TEST-ONLY: rt_trace.cuh ray_hit (which rt_ray_kernel calls per lane) for n rays of 8 floats each, written like the
// kernel writes the outputs.  flags: bit 31 selects the FILTER walk, bit 30 the CULL walk (as aov_hostsim), else the
// direct loops.  Returns 0 on success.
extern "C" int hostsim_trace_rays(const char* scene_text, size_t n, const float* rays, uint32_t flags, float* depth,
                                  float* position, float* normal, float* albedo, int32_t* prim)
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
        AovRecord r;
        if (flags & 0x40000000u)      r = ray_hit<RT_SPH_CULL, true>(G, G.sph_filter, G.sph_r2, cv, G.tri_plane, r0, r1, 1.0f);
        else if (flags & 0x80000000u) r = ray_hit<RT_SPH_FILTER, true>(G, G.sph_filter, G.sph_r2, cv, G.tri_plane, r0, r1, 1.0f);
        else if (G.n_tri_pad)         r = ray_hit<RT_SPH_DIRECT, true>(G, G.sph, nullptr, cv, G.tri_plane, r0, r1, 1.0f);
        else                          r = ray_hit<RT_SPH_DIRECT, false>(G, G.sph, nullptr, cv, G.tri_plane, r0, r1, 1.0f);
        depth[i] = r.t;
        position[3 * i] = r.pos.x; position[3 * i + 1] = r.pos.y; position[3 * i + 2] = r.pos.z;
        normal[3 * i] = r.n.x; normal[3 * i + 1] = r.n.y; normal[3 * i + 2] = r.n.z;
        albedo[3 * i] = r.albedo.x; albedo[3 * i + 1] = r.albedo.y; albedo[3 * i + 2] = r.albedo.z;
        prim[i] = r.prim;
    }
    return 0;
}
