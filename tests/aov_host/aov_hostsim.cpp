// aov_hostsim.cpp — TEST-ONLY: compiles the device header csrc/rt_trace.cuh (exact policy) with g++ and drives the
// first-hit kernel's per-pixel helper on the host, so that it can be checked against the CPU reference
// (aov_reference.c) on a machine without a GPU.  It is NOT part of the product and is never loaded by the package:
// only tests/test_aov.py loads it.
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

// TEST-ONLY: the first-hit kernel's per-pixel helper (rt_trace.cuh first_hit, which rt_aov_kernel calls per lane) for
// every pixel of a W x H frame, written like the kernel writes the buffers.  flags: bit 0 RT_FLAG_FIXED_JITTER; bit 31
// selects the FILTER walk, bit 30 the CULL walk (as tests/hostsim hostsim_render), else the direct loops.  Returns 0 on success.
extern "C" int hostsim_primary_hits(const char* scene_text, const float cam12[12], uint32_t W, uint32_t H, uint32_t seed,
                                    int32_t sample_begin, uint32_t flags, float* depth, float* position, float* normal,
                                    float* albedo, int32_t* prim)
{
    using namespace rt;
    ParseResult pr = parse_input(scene_text, std::strlen(scene_text));
    if (pr.error != ParseError::Ok) return (int)pr.error;
    const World::Packed& pk = pr.world->packed();
    RtSceneView G = pk.view(pk.blob.data());
    if ((flags & 0x40000000u) && G.n_groups == 0) return 100;      // the world has no block C (< 64 spheres)

    RtAovParams A{};
    std::memcpy(&A.camera, cam12, sizeof(float) * 12);
    A.width = W; A.height = H; A.wm1 = (float)(W - 1u); A.hm1 = (float)(H - 1u);
    A.seed = seed; A.sample_begin = sample_begin; A.flags = flags & RT_FLAG_FIXED_JITTER; A.one = 1.0f;
    CullView cv{G.cull_bound, G.cull_sph, G.cull_r2, G.cull_orig, G.n_groups};
    for (uint32_t row = 0; row < H; ++row)
        for (uint32_t x = 0; x < W; ++x) {
            AovRecord r;
            if (flags & 0x40000000u)      r = first_hit<false, RT_SPH_CULL, true>(A, G, G.sph_filter, G.sph_r2, cv, G.tri_plane, x, row);
            else if (flags & 0x80000000u) r = first_hit<false, RT_SPH_FILTER, true>(A, G, G.sph_filter, G.sph_r2, cv, G.tri_plane, x, row);
            else if (G.n_tri_pad)         r = first_hit<false, RT_SPH_DIRECT, true>(A, G, G.sph, nullptr, cv, G.tri_plane, x, row);
            else                          r = first_hit<false, RT_SPH_DIRECT, false>(A, G, G.sph, nullptr, cv, G.tri_plane, x, row);
            const size_t i = (size_t)row * W + x;
            depth[i] = r.t;
            position[3 * i] = r.pos.x; position[3 * i + 1] = r.pos.y; position[3 * i + 2] = r.pos.z;
            normal[3 * i] = r.n.x; normal[3 * i + 1] = r.n.y; normal[3 * i + 2] = r.n.z;
            albedo[3 * i] = r.albedo.x; albedo[3 * i + 1] = r.albedo.y; albedo[3 * i + 2] = r.albedo.z;
            prim[i] = r.prim;
        }
    return 0;
}
