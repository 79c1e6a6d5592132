// rt_types.h — plain data shared by the host layer and the CUDA kernels.
//
// Layout in HBM (one contiguous, 16-byte aligned "scene blob" per device, built once per
// load_world / World::new and never touched by the render loop again):
//
//   block A (staged into shared memory by the direct kernels)
//   [ sph       : float4 x Sp]  {cx, cy, cz, r*r} of consecutive spheres in PAIRS, two float4 per pair:
//                               {x0, x1, y0, y1} {z0, z1, r0*r0, r1*r1} (operands of FMUL2 / FADD2)          hot
//   [ tri_plane : float4 x Tp]  {n.x, n.y, n.z, n.v0} of consecutive triangles in PAIRS: {nx0, nx1, ny0, ny1}
//                               {nz0, nz1, w0, w1}                                                          hot
//   block B (staged instead of A by the FILTER kernels, large sphere counts)
//   [ sph_filter: float4 x Sp]  the filter records {cx, cy, cz, w = c.c - r*r - margin} of consecutive spheres in
//                               PAIRS, two float4 per pair: {x0, x1, y0, y1} {z0, z1, -w0, -w1} — the operand layout of
//                               the two-wide FMAs (FFMA2)                   hot  (rt_trace.cuh, sphere_filter_group_n)
//   [ tri_plane : float4 x Tp]  (same as in block A)              hot
//   [ sph_r2    : float  x Sp]  r*r                               warm (filter survivors only)
//   block C (staged instead of A/B by the CULL kernels: RT_FLAG_GROUP_CULL, an opt-in mode)
//   [ cull_bound: float4 x Gc]  bounding sphere of a group of 8 spheres: {cB.xyz, wB}    hot
//   [ cull_sph  : float4 x 9Gc] the spheres in spatial (Morton) order, 8 filter records
//                               {c.xyz, c.c - r*r - margin} per group + one float4 {gB,0,0,0};
//                               the 144-byte group stride spreads per-lane group reads over the banks   hot
//   [ tri_plane : float4 x Tp]  (same as in block A)                                  hot
//   [ cull_r2   : float  x 8Gc] r*r in the same order                                 warm
//   [ cull_orig : u32    x 8Gc] list index of each sphere (hit-test order = tie-break order)  warm
//   then
//   [ tri_cull  : float4 x 5Tp/2]  per PAIR of triangles {G2.xyz, g2}, {G0.xyz, g0}, K — approximate barycentric
//                               gradients for the conservative edge-stage reject — as {G2x0,G2x1,G2y0,G2y1}
//                               {G2z0,G2z1,g2_0,g2_1} {G0x0,..} {G0z0,..,g0_1} {K0,K1,0,0}   warm (plane-stage survivors)
//   [ tri_v     : float4 x 3T]  {v_k.xyz, stored_normal[k]}       cool (reject survivors)
//   [ info      : 32 B   x P ]  RtPrimInfo                        cold (one gather per hit), P = S+T
//
// Sp = S rounded up to a multiple of RT_SPHERE_GROUP, Tp = T rounded up to a multiple of
// RT_TRI_GROUP; the padding entries are all-NaN, which can never be hit (every comparison
// with NaN is false), so the closest-hit loops run in whole groups without remainder loops.
//
// This is the SoA split the reference author sketches in raytracer/TODO.txt:27-39: the
// closest-hit loop reads 16 B per primitive and nothing else.
#pragma once
#include <stddef.h>
#include <stdint.h>

// materials.rs:7-12
enum RtMaterialType : uint32_t {
    RT_MAT_DIFFUSE    = 0,
    RT_MAT_METAL      = 1,
    RT_MAT_DIELECTRIC = 2,
    RT_MAT_EMISSION   = 3,
};

struct RtVec3 { float x, y, z; };

// camera.rs:8-15
struct RtCameraData {
    RtVec3 origin;
    RtVec3 lower_left_corner;
    RtVec3 horizontal;
    RtVec3 vertical;
};

struct RtFloat4 { float x, y, z, w; };

#define RT_SPHERE_GROUP 8u
#ifndef RT_FILTER_GROUP
#define RT_FILTER_GROUP 8u     /* spheres per group of the FILTER kernels (a multiple of RT_SPHERE_GROUP) */
#endif
#define RT_FILTER_FROM  64u    /* sphere lists of at least this many run the FILTER kernels */
/* How the spheres are walked (template parameter SPH of the kernels) */
#define RT_SPH_DIRECT 0   /* the reference's test for every sphere */
#define RT_SPH_FILTER 1   /* conservative 8-instruction filter first */
#define RT_SPH_CULL   2   /* bounding spheres of groups first, then the filter, then the reference's test */
/* constants of the group bound test (rt_trace.cuh cull_spheres, rt_scene.cpp build_cull_block) */
#define RT_CULL_B   3.5e-3f                 /* >= sqrt(189 * 2^-24): growth of a member's effective radius with |o|+|c|+r */
#define RT_CULL_M   3.0517578125e-05f       /* 2^-15: margin of the bound test's own evaluation */
#define RT_TRI_GROUP    2u

// Everything the shading step needs about the primitive that was hit: one 32-byte record,
// fetched with two 16-byte loads.
struct RtPrimInfo {
    float    r, g, b;       // Color (alpha == 1)
    float    param;         // Metal: fuzz, Dielectric: ir
    uint32_t type;          // RT_MAT_*
    float    inv_param;     // Dielectric: 1.0f / ir (materials.rs:69, evaluated once on the host)
    float    radius;        // spheres: radius (common.rs:95 divides by it); triangles: 1
    float    pad;
};

// Device- or host-resident view of a packed scene (pointers into the blob).
struct RtSceneView {
    const RtFloat4*   sph;        // [n_sph_pad]  block A
    const RtFloat4*   tri_plane;  // [n_tri_pad]  block A
    const RtFloat4*   sph_filter; // [n_sph_pad]  block B (followed by tri_plane again, then sph_r2)
    const float*      sph_r2;     // [n_sph_pad]  block B
    const RtFloat4*   cull_bound; // [n_groups]     block C
    const RtFloat4*   cull_sph;   // [9*n_groups]   block C (followed by tri_plane again)
    const float*      cull_r2;    // [8*n_groups]
    const uint32_t*   cull_orig;  // [8*n_groups]
    const RtFloat4*   tri_cull;   // [3T]
    const RtFloat4*   tri_v;      // [3T]
    const RtPrimInfo* info;       // [S+T]
    uint32_t          n_sph;
    uint32_t          n_sph_pad;  // multiple of RT_SPHERE_GROUP
    uint32_t          n_tri;
    uint32_t          n_tri_pad;  // multiple of RT_TRI_GROUP
    uint32_t          n_groups;   // block C: groups of 8 spheres (0: the world has no block C)
    uint32_t          pad;
};

// Row-tile sharding.  The frame's tiles (tile_rows image rows each, top to bottom) are dealt to
// the shards in stripes of `count` consecutive tiles, alternately forwards and backwards
// (boustrophedon): the j-th tile of shard `index` is tile j*count + (j even ? index : count-1-index).
// A plain round-robin gives the last shard the lowest tile of EVERY stripe, and cost grows
// towards the ground; the alternation cancels such a gradient to first order.  (Measured on C4,
// 4 GPUs: 131.4-135.8 ms per rank for the 16 passes, the spread being the one tile rank 0 has less.)
#if defined(__CUDACC__)
__host__ __device__
#endif
inline uint32_t rt_shard_tile(uint32_t index, uint32_t count, uint32_t j)
{
    return j * count + ((j & 1u) ? count - 1u - index : index);
}

// Flags of RtFrameParams::flags
enum : uint32_t {
    RT_FLAG_FIXED_JITTER = 1u << 0,   // sub-pixel offset (0.5, 0.5); no jitter draws
    RT_FLAG_ACCUM_IN     = 1u << 1,   // continue from the float4 accumulator (progressive pass)
    RT_FLAG_ACCUM_OUT    = 1u << 2,   // write the float4 accumulator back
    RT_FLAG_NO_RESOLVE   = 1u << 3,   // skip the RGBA8 pack (intermediate progressive pass)
    RT_FLAG_COMPACT_OUT  = 1u << 4,   // out/accum hold only this shard's tiles, packed
    RT_FLAG_GROUP_CULL   = 1u << 6,   // run the CULL kernels (block C): same hits, fewer sphere tests
    RT_FLAG_SAMPLE_ITEMS = 1u << 5,   // work items are (pixel, sample) pairs; colours go to `samples`, the
                                      // ordered sum + resolve is done by rt_resolve_samples_kernel
    RT_FLAG_RESOLVE_EACH_PASS = 1u << 7,   // fused progressive passes: store the resolved pixel after every pass
};

// Division of a 32-bit unsigned by a launch constant without the divide (Granlund & Montgomery's round-up form:
// exact for EVERY n < 2^32 and every d in [1, 2^31]): with l = ceil(log2 d), mul = floor(2^32 (2^l - d) / d) + 1,
//     t = hi32(mul * n),  n / d = (t + ((n - t) >> min(l, 1))) >> max(l - 1, 0).
// Five integer instructions where the compiler's own expansion of `n / d` (float reciprocal, two corrections) takes ~20;
// the slot decode of the render kernel divides twice per pixel (rt_kernels.cuh, decode_slot).
struct RtDivisor { uint32_t d, mul, sh1, sh2; };
#if defined(__CUDACC__)
__host__ __device__
#endif
inline RtDivisor rt_divisor(uint32_t d)
{
    RtDivisor k;
    k.d = d;
    uint32_t l = 0;
    while (l < 32u && (1ull << l) < d) ++l;                              // ceil(log2 d); d = 0 is never divided by
    k.mul = (uint32_t)((((1ull << l) - d) << 32) / (d ? d : 1u)) + 1u;
    k.sh1 = l < 1u ? l : 1u;
    k.sh2 = l > 0u ? l - 1u : 0u;
    return k;
}
#if defined(__CUDACC__)
__host__ __device__
#endif
inline uint32_t rt_div(uint32_t n, const RtDivisor& k)
{
#if defined(__CUDA_ARCH__)
    const uint32_t t = __umulhi(k.mul, n);
#else
    const uint32_t t = (uint32_t)(((unsigned long long)k.mul * n) >> 32);
#endif
    return (t + ((n - t) >> k.sh1)) >> k.sh2;
}

// One work queue of a launch.  Queue 0 is the launch's own shard; further entries are the shards
// of OTHER GPUs rendering the same frame, whose work counter (and float4 sums) live in their
// memory and are reached through peer / CUDA-IPC mappings: when a warp finds its own queue empty
// it takes slabs from the other queues (atomicAdd at system scope over NVLink) — the tail of the
// frame is stolen by whichever GPU is free (SURVEY.md 8e).
#define RT_MAX_QUEUES 8u
struct RtQueue {
    unsigned int* work_counter;   // next unassigned slot of this shard (reset by its owner before every frame)
    RtFloat4*     accum;          // this shard's float4 sums (fused passes), indexed like `out`
    uint32_t      tile_first;     // shard index: the queue's tiles are rt_shard_tile(tile_first, tile_stride, j)
    uint32_t      n_tiles;
};

// Everything one render launch needs (passed by value as a __grid_constant__).
struct RtFrameParams {
    RtCameraData camera;
    float    wm1, hm1;       // (W-1) as f32, (H-1) as f32: the divisors of common.rs:335-336
    uint32_t width, height;
    int32_t  spp;            // samples traced per pixel and pass by this launch (common.rs:334)
    int32_t  depth;          // max_ray_bounces (common.rs:267)
    int32_t  sample_begin;   // index of this launch's first sample (progressive passes)
    int32_t  resolve_spp;    // divisor of the resolve (common.rs:345-348)
    uint32_t seed;
    uint32_t flags;
    // Row-tile sharding: this launch renders image-row tiles
    //   rt_shard_tile(tile_first, tile_stride, j), j = 0 .. n_tiles-1   (tile_rows rows each).
    uint32_t tile_rows, tile_first, tile_stride, n_tiles;
    uint32_t reserve;        // pixel slots a warp takes per atomicAdd (multiple of 32)
    // Progressive passes fused into ONE launch (1 = a plain frame).  The work space is pass-major:
    // slot s belongs to pass s / (slots per pass) and traces samples sample_begin + pass*spp ...
    // A pixel's pass p starts from the float4 sums its pass p-1 left in `accum` (whichever lane,
    // warp or GPU traced it): the alpha channel of the sums counts the samples (1 + p*spp), so the
    // 16-byte record carries its own "ready" tag, and a lane whose pixel is not ready yet simply
    // retries in its next loop iteration.  No drain between passes, one ramp-up per frame.
    uint32_t passes;
    float    one;            // 1.0f, as a value the compiler cannot see: multiplier of the exact policy's two-wide sums
                             // (rt_trace.cuh f2_add1) — set by the host, never anything else
    uint32_t pad_one;
    uint32_t* out;           // RGBA8 as u32, full frame or compact (RT_FLAG_COMPACT_OUT)
    RtFloat4* accum;         // optional float4 sums, same indexing as out
    unsigned long long* ray_counter;   // += number of World::hit calls
    unsigned int* work_counter;        // zeroed before launch
    unsigned int* steal_counter;       // += slots taken from other shards' queues (may be null)
    // RT_FLAG_SAMPLE_ITEMS: colour of sample s of the pixel with output index i at samples[s*sample_stride + i]
    RtFloat4* samples;
    uint32_t  sample_stride;
    // Tile completion (optional): tile_done[t] counts the finished pixels of image tile t; the lane that
    // completes a tile publishes tile_flags[t] = tile_epoch (host-mapped memory), after a system-scope fence, so
    // that the host can hand the tile's rows on while the kernel is still rendering the rest of the frame.
    unsigned int* tile_done;
    unsigned int* tile_flags;
    uint32_t  tile_epoch;
    uint32_t  pad_tile;
    // divisors of the slot decode (set by the host next to width / tile_rows): sub-tiles of 8x4 pixels per strip of
    // tile_rows rows, and per row of sub-tiles
    RtDivisor div_chunks_per_strip, div_subtiles_x;
    uint32_t  n_queues;      // >= 1
    RtQueue   queues[RT_MAX_QUEUES];   // [0] = the launch's own shard (work_counter / accum above), then the peers
};

// Everything one first-hit launch needs (rt_aov_kernel, passed by value as a __grid_constant__): the camera ray of
// sample `sample_begin` of every pixel of a width x height frame, traced once, and World::hit's record written to
// whichever of the five buffers is non-null (image row 0 = top, row-major, like the RGBA8 frame).
struct RtAovParams {
    RtCameraData camera;
    float    wm1, hm1;       // (W-1) as f32, (H-1) as f32: the divisors of common.rs:335-336
    uint32_t width, height;
    uint32_t seed;
    int32_t  sample_begin;   // the sample whose camera ray is traced
    uint32_t flags;          // RT_FLAG_FIXED_JITTER (the walk is a template parameter of the kernel)
    float    one;            // 1.0f, as a value the compiler cannot see (RtFrameParams::one)
    float*   depth;          // [H][W]     HitRecord.t, +inf on a miss
    float*   position;       // [H][W][3]  Ray::at(t), 0 on a miss
    float*   normal;         // [H][W][3]  hit normal, 0 on a miss
    float*   albedo;         // [H][W][3]  material colour, the sky colour of the ray on a miss
    int32_t* prim;           // [H][W]     sphere i -> i, triangle j -> S + j, -1 on a miss
};

// Everything one denoise call needs (rt_denoise.cu): the edge-avoiding a-trous filter of a frame's colour sums, guided
// by the first-hit buffers.  Inputs and outputs are row-major, top row first, like the RGBA8 frame.
struct RtDenoiseParams {
    const RtFloat4* accum;      // [H][W]     colour sums (RT_OPT_ACCUM_OUT)
    const float*    normal;     // [H][W][3]  first-hit guides (rt_render_aov_device)
    const float*    position;   // [H][W][3]
    const float*    albedo;     // [H][W][3]
    const int32_t*  prim;       // [H][W]     < 0: a miss pixel
    uint32_t*       pixels;     // [H][W]     RGBA8 out, or null
    RtFloat4*       color;      // [H][W]     float4 out, or null
    RtFloat4*       e[2];       // [H][W]     scratch: the demodulated colour, ping-pong
    RtFloat4*       gn;         // [H][W]     scratch: normal, miss flag (w = 1 on a miss)
    RtFloat4*       gx;         // [H][W]     scratch: position
    uint32_t        width, height;
    uint32_t        iterations; // 1..10
    float           k;          // 1.0f / spp
    float           sc, sn, sx; // 1 / ((16 sigma) sigma) of colour, normal and plane distance
};

// Everything one ray-query launch needs (rt_ray_kernel, passed by value as a __grid_constant__): n caller-supplied rays,
// each two float4 {origin, t_max} {direction, reserved} (RtRay of raytracer_b200.h, 16-byte aligned), and World::hit's
// record of ray i written to element i of whichever of the five buffers is non-null (DESIGN.md §13).
struct RtRayParams {
    const RtFloat4* rays;    // [n][2]
    uint32_t n;              // 1 .. 2^31 - 1
    float    one;            // 1.0f, as a value the compiler cannot see (RtFrameParams::one)
    float*   depth;          // [n]     HitRecord.t, +inf on a miss, NaN for an invalid ray
    float*   position;       // [n][3]  Ray::at(t), 0 on a miss or an invalid ray
    float*   normal;         // [n][3]  hit normal, 0 on a miss or an invalid ray
    float*   albedo;         // [n][3]  material colour, the sky colour of the ray on a miss, 0 for an invalid ray
    int32_t* prim;           // [n]     sphere i -> i, triangle j -> S + j, -1 on a miss, -2 for an invalid ray
};

// Everything one occlusion-query launch needs (rt_occlusion_kernel, a __grid_constant__): n rays laid out as for
// RtRayParams, and one byte per ray (DESIGN.md §14).
struct RtOcclusionParams {
    const RtFloat4* rays;    // [n][2]
    uint32_t n;              // 1 .. 2^31 - 1
    float    one;            // 1.0f, as a value the compiler cannot see (RtFrameParams::one)
    uint8_t* occluded;       // [n]     1: World::hit returns a hit, 0: it returns none, 2: an invalid ray
};

// Everything one temporal-accumulation call needs (rt_temporal.cu, DESIGN.md §15): a frame's colour sums blended with
// the colour history of the previous frame, looked up where each pixel's surface was in the previous camera.  Inputs
// and outputs are row-major, top row first, like the RGBA8 frame.
#define RT_TEMPORAL_NO_HISTORY  0u   // every pixel gets its mean
#define RT_TEMPORAL_SAME_CAMERA 1u   // the previous camera equals this one bit for bit: the only tap is the pixel itself
#define RT_TEMPORAL_REPROJECT   2u   // the bilinear 2x2 taps around the pixel's projection into the previous camera
struct RtTemporalParams {
    const RtFloat4* accum;          // [H][W]     colour sums of spp samples (RT_OPT_ACCUM_OUT)
    const float*    position;       // [H][W][3]  first-hit guides of this frame (rt_render_aov_device)
    const float*    normal;         // [H][W][3]
    const int32_t*  prim;           // [H][W]     < 0: a miss pixel
    const RtFloat4* prev_color;     // [H][W]     the previous frame's colour output (null without history)
    const float*    prev_length;    // [H][W]     its history length, in samples
    const float*    prev_position;  // [H][W][3]  the previous frame's guides
    const float*    prev_normal;    // [H][W][3]
    const int32_t*  prev_prim;      // [H][W]
    RtFloat4*       color;          // [H][W]     float4 out: the blended mean, alpha 1
    float*          length;         // [H][W]     out: the samples behind it
    uint32_t*       pixels;         // [H][W]     RGBA8 out, or null
    uint32_t        width, height;
    uint32_t        mode;           // RT_TEMPORAL_*
    float           k;              // 1.0f / spp
    float           spp;            // (float)spp
    float           max_history;    // (float)max_history
    float           normal_cos;     // a tap's normal must satisfy dot(n_p, n_q) >= normal_cos
    float           plane_tol;      // and its position |dot(n_p, x_q - x_p)| <= plane_tol
    float           wm1, hm1;       // (float)(W - 1), (float)(H - 1)
    float           fw, fh;         // (float)W, (float)H
    // the projection into the previous camera (origin o', lower-left corner L', horizontal h', vertical v'), computed
    // once per call by tp_setup_projection: a = L' - o', cn = cross(h', v'), cs = cross(v', a), ct = cross(a, h')
    RtVec3          prev_origin;
    RtVec3          cn, cs, ct;
    float           det;            // dot(a, cn)
};

struct RtFloat2 { float x, y; };

// Everything one SVGF call needs (rt_svgf.cu, DESIGN.md §16): the temporal stage of §15 carrying the demodulated colour
// and the first two luminance moments, a variance estimate per pixel, and the a-trous filter of §12 with its colour
// weight scaled by that variance.  Inputs and outputs are row-major, top row first, like the RGBA8 frame.
struct RtSvgfParams {
    // the history lookup of §15: accum, this frame's position / normal / prim, the previous frame's guides,
    // prev_color = its illum output and prev_length = its length output, mode, k, spp, max_history, normal_cos,
    // plane_tol and the projection constants; its color, length and pixels outputs are not used
    RtTemporalParams t;
    const float*    albedo;         // [H][W][3]  first-hit albedo of this frame
    const RtFloat2* prev_moments;   // [H][W]     the previous frame's moments output (null without history)
    RtFloat4*       illum;          // [H][W]     out: the first a-trous iteration's demodulated colour (next history)
    RtFloat2*       moments;        // [H][W]     out: the temporal luminance moments (l, l*l)
    float*          length;         // [H][W]     out: the samples behind them
    uint32_t*       pixels;         // [H][W]     RGBA8 out, or null
    RtFloat4*       color;          // [H][W]     float4 out, or null
    RtFloat4*       e[2];           // [H][W]     scratch: demodulated colour, luminance in w, ping-pong
    float*          var[2];         // [H][W]     scratch: luminance variance, ping-pong
    RtFloat4*       gn;             // [H][W]     scratch: normal, miss flag (w = 1 on a miss)
    RtFloat4*       gx;             // [H][W]     scratch: position
    uint32_t        iterations;     // 1..10
    float           spp4;           // 4.0f * (float)spp: a history this long has its own variance
    float           ql;             // (16 sigma_luminance) sigma_luminance
    float           sn, sx;         // 1 / ((16 sigma) sigma) of normal and plane distance
};
