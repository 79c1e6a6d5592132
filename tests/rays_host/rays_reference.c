/*
 * rays_reference.c — TEST INFRASTRUCTURE ONLY: the CPU reference of the ray-query records (rt_trace_rays_device),
 * built on the public API of the oracle (oracle/rt_oracle.h; linked against oracle/build/librt_oracle.so, never into
 * the product).
 *
 * rays: n records of 8 floats {origin[3], t_max, direction[3], reserved}.  Per ray, in the order of the semantics of
 * include/raytracer_b200.h:
 *   1. the domain check — no NaN among the seven floats, finite origin with |o.c| <= 2^40, and s = (dx*dx + dy*dy) +
 *      dz*dz in [2^-100, 2^100] (unfused: this file is compiled with -ffp-contract=off); an invalid ray gets prim -2,
 *      depth NaN (bits 0x7fffffff) and zeros;
 *   2. d = orc_normalize(direction) (NVec3::new, maths.rs:111-118);
 *   3. orc_world_hit(o, d) — World::hit with t_max = +inf — then the caller's t_max: a sphere hit survives when
 *      t < t_max, a triangle hit when t <= t_max, else the ray misses;
 *   4. the record of the first-hit buffers (aov_reference.c): depth t (+inf on a miss), position and normal of the
 *      hit record (0 on a miss), albedo the material's colour (Dielectric 1,1,1) or on a miss the sky colour of d,
 *      prim sphere i -> i, triangle j -> n_spheres + j, -1 on a miss.
 * Any output may be NULL.  Returns 0.
 */
#include <math.h>
#include <stddef.h>
#include <stdint.h>
#include <string.h>

#include "../../oracle/rt_oracle.h"

static int in_domain(const float *r)
{
    const float lim = 1099511627776.0f;                                 /* 2^40 */
    for (int c = 0; c < 3; ++c)
        if (!(fabsf(r[c]) <= lim)) return 0;                            /* NaN and inf fail */
    if (r[3] != r[3]) return 0;                                         /* t_max NaN; +-inf are valid */
    const float s = r[4] * r[4] + r[5] * r[5] + r[6] * r[6];
    return s >= 0x1p-100f && s <= 0x1p100f;                             /* NaN fails */
}

int rays_reference(const orc_world *w, size_t n, const float *rays, float *depth, float *position, float *normal,
                   float *albedo, int32_t *prim)
{
    const size_t        n_spheres = orc_world_sphere_count(w);
    const orc_sphere   *spheres   = orc_world_spheres(w);
    const orc_triangle *triangles = orc_world_triangles(w);
    for (size_t i = 0; i < n; ++i) {
        const float *r   = rays + 8 * i;
        float        t   = INFINITY;
        orc_vec3     pos = { 0.0f, 0.0f, 0.0f }, nrm = { 0.0f, 0.0f, 0.0f }, alb = { 0.0f, 0.0f, 0.0f };
        int64_t      p   = -1;
        if (!in_domain(r)) {
            const uint32_t nan_bits = 0x7fffffffu;
            memcpy(&t, &nan_bits, 4);
            p = -2;
        } else {
            const orc_vec3 o = { r[0], r[1], r[2] }, a = { r[4], r[5], r[6] };
            const float    t_max = r[3];
            const orc_vec3 d     = orc_normalize(a);
            int hit = orc_world_hit(w, o, d, &t, &pos, &nrm, &p);
            if (hit && !(p < (int64_t)n_spheres ? t < t_max : t <= t_max)) hit = 0;      /* the caller's t_max */
            if (hit) {
                const orc_material *m = p < (int64_t)n_spheres ? &spheres[p].material
                                                               : &triangles[p - (int64_t)n_spheres].material;
                if (m->type == ORC_DIELECTRIC) { alb.x = 1.0f; alb.y = 1.0f; alb.z = 1.0f; }
                else                           { alb.x = m->r; alb.y = m->g; alb.z = m->b; }
            } else {
                /* common.rs:278-280, as aov_reference.c: lerp((1,1,1), (0.5,0.7,1), t) of the ray's unit direction */
                const float st = 0.5f * (orc_normalize(d).y + 1.0f), mt = 1.0f - st;
                alb.x = 1.0f * mt + 0.5f * st;
                alb.y = 1.0f * mt + 0.7f * st;
                alb.z = 1.0f * mt + 1.0f * st;
                t = INFINITY;
                p = -1;
                pos.x = pos.y = pos.z = 0.0f;
                nrm.x = nrm.y = nrm.z = 0.0f;
            }
        }
        if (depth) depth[i] = t;
        if (position) { position[3 * i] = pos.x; position[3 * i + 1] = pos.y; position[3 * i + 2] = pos.z; }
        if (normal) { normal[3 * i] = nrm.x; normal[3 * i + 1] = nrm.y; normal[3 * i + 2] = nrm.z; }
        if (albedo) { albedo[3 * i] = alb.x; albedo[3 * i + 1] = alb.y; albedo[3 * i + 2] = alb.z; }
        if (prim) prim[i] = (int32_t)p;
    }
    return 0;
}
