/*
 * aov_reference.c — TEST INFRASTRUCTURE ONLY: the CPU reference of the first-hit buffers, built on the public API of
 * the oracle (oracle/rt_oracle.h; linked against oracle/build/librt_oracle.so, never into the product).
 *
 * For every pixel the ONE camera ray of sample `sample_begin` that orc_ray_trace (PER_SAMPLE mode) traces first —
 * common.rs:335-337: u drawn first, (col + xi1)/(W-1) and (row + xi2)/(H-1) as f32 divides (xi = 0.5, no draws, when
 * fixed_jitter != 0), orc_cast_ray — and orc_world_hit's record for it, top row first:
 *   depth [H*W]: t (+inf on a miss);  position / normal [H*W*3]: the hit record's (0 on a miss);
 *   albedo [H*W*3]: the hit material's colour, Dielectric 1,1,1 (materials.rs:95); on a miss the sky colour of the
 *   ray, common.rs:276-281, as the oracle's ray_color computes it;  prim [H*W]: sphere i -> i, triangle j ->
 *   n_spheres + j (-1 on a miss).
 * Only image rows [image_row_begin, image_row_end) of the full-frame arrays are written (a band of the frame is exactly
 * that band: every pixel has its own sample stream).  Any output may be NULL.  Returns 0.
 */
#include <math.h>
#include <stddef.h>
#include <stdint.h>

#include "../../oracle/rt_oracle.h"

int aov_primary_hits_rows(const orc_world *w, const orc_camera *camera, size_t width, size_t height,
                          size_t image_row_begin, size_t image_row_end, uint32_t seed, int32_t sample_begin,
                          int32_t fixed_jitter, float *depth, float *position, float *normal, float *albedo,
                          int32_t *prim)
{
    const size_t        n_spheres = orc_world_sphere_count(w);
    const orc_sphere   *spheres   = orc_world_spheres(w);
    const orc_triangle *triangles = orc_world_triangles(w);
    if (image_row_end > height) image_row_end = height;
    for (size_t image_row = image_row_begin; image_row < image_row_end; ++image_row) {
        const size_t row = height - 1 - image_row;                 /* :351 */
        for (size_t column = 0; column < width; ++column) {
            const size_t i = image_row * width + column;
            uint32_t rng = orc_sample_seed(seed, (uint32_t)(row * width + column), (uint32_t)sample_begin);
            float ju = fixed_jitter ? 0.5f : orc_random_f32(&rng);   /* :335, u first */
            float u  = ((float)column + ju) / (float)(width - 1);
            float jv = fixed_jitter ? 0.5f : orc_random_f32(&rng);   /* :336 */
            float v  = ((float)row + jv) / (float)(height - 1);
            orc_vec3 o, d;
            orc_cast_ray(camera, u, v, &o, &d);
            float    t   = INFINITY;
            orc_vec3 pos = { 0.0f, 0.0f, 0.0f }, nrm = { 0.0f, 0.0f, 0.0f }, alb;
            int64_t  p   = -1;
            if (orc_world_hit(w, o, d, &t, &pos, &nrm, &p)) {
                const orc_material *m = p < (int64_t)n_spheres ? &spheres[p].material
                                                               : &triangles[p - (int64_t)n_spheres].material;
                if (m->type == ORC_DIELECTRIC) { alb.x = 1.0f; alb.y = 1.0f; alb.z = 1.0f; }
                else                           { alb.x = m->r; alb.y = m->g; alb.z = m->b; }
            } else {
                /* :278-280: lerp((1,1,1), (0.5,0.7,1), t) = a*(1-t) + b*t, as in the oracle's ray_color */
                const float st = 0.5f * (orc_normalize(d).y + 1.0f), mt = 1.0f - st;
                alb.x = 1.0f * mt + 0.5f * st;
                alb.y = 1.0f * mt + 0.7f * st;
                alb.z = 1.0f * mt + 1.0f * st;
                t = INFINITY;
                p = -1;
            }
            if (depth) depth[i] = t;
            if (position) { position[3 * i] = pos.x; position[3 * i + 1] = pos.y; position[3 * i + 2] = pos.z; }
            if (normal) { normal[3 * i] = nrm.x; normal[3 * i + 1] = nrm.y; normal[3 * i + 2] = nrm.z; }
            if (albedo) { albedo[3 * i] = alb.x; albedo[3 * i + 1] = alb.y; albedo[3 * i + 2] = alb.z; }
            if (prim) prim[i] = (int32_t)p;
        }
    }
    return 0;
}
