/*
 * raytracer_b200.h — additive C ABI of the B200-native render path.  Nothing here exists
 * in the reference; each entry cites the reference code whose behaviour it exposes.
 * Plain pointers and sizes only (no torch / CUDA types in the signatures); device pointers
 * and streams travel as void*.
 */
#ifndef RAYTRACER_B200_H
#define RAYTRACER_B200_H

#include "raytracer.h"

#ifdef __cplusplus
extern "C" {
#endif

#define RT_B200_ABI_VERSION 2u   /* 2: RtRenderStats and RtRenderOptions grew (fused passes, work stealing) */

/* RtRenderOptions::flags */
#define RT_OPT_FIXED_JITTER 0x1u  /* deterministic mode: sub-pixel offset (0.5,0.5), no jitter draws */
#define RT_OPT_FAST_MATH    0x2u  /* relaxed-arithmetic kernel: FMA/rsqrt, statistically equal only */
#define RT_OPT_ACCUM_IN     0x4u  /* continue from device_accum (progressive pass) */
#define RT_OPT_ACCUM_OUT    0x8u  /* store the float4 sums back to device_accum */
#define RT_OPT_NO_RESOLVE   0x10u /* skip the RGBA8 pack (intermediate progressive pass) */
#define RT_OPT_PIXEL_ITEMS  0x40u /* scheduling only: a lane always owns a whole pixel */
#define RT_OPT_SAMPLE_ITEMS 0x80u /* scheduling only: work items are single samples, summed in order by a
                                     second kernel (default: chosen from the scene and frame size) */
#define RT_OPT_GROUP_CULL   0x100u /* acceleration (SURVEY 8f-4), opt-in and reported separately: spheres are kept in
                                      spatial groups of 8 with conservative bounding spheres; a ray tests only the
                                      groups it can touch.  Same pixels and ray counts, fewer sphere tests.
                                      Worlds with fewer than 64 spheres ignore it. */
#define RT_OPT_RESOLVE_EACH_PASS 0x200u /* passes > 1: refresh the RGBA8 frame after every pass, not only the last */
#define RT_OPT_NO_STEAL      0x400u /* peer_queues given: no cross-GPU work stealing (static tile deal only) */
#define RT_OPT_ROW_GATHER    0x800u /* rt_render_device with RT_OPT_FULL_FRAME_OUT when device_pixels is a frame in ANOTHER
                                       GPU's memory: the shard is rendered into a local, zeroed frame and a small second kernel
                                       moves every pixel found there across as 16-byte vectors, instead of one 4-byte store
                                       per pixel over NVLink.  (A zero word means "not rendered here": alpha is always 255.) */
#define RT_OPT_FULL_FRAME_OUT 0x20u /* rt_render_device with shard_count > 1: device_pixels / device_accum are
                                       FULL width*height frames (e.g. another GPU's frame mapped through CUDA IPC
                                       or peer access); this shard's tiles are stored at their frame offsets */

/* materials.rs:7-12 */
#define RT_MATERIAL_DIFFUSE    0u
#define RT_MATERIAL_METAL      1u
#define RT_MATERIAL_DIELECTRIC 2u
#define RT_MATERIAL_EMISSION   3u

typedef struct RtRenderStats {
  uint64_t rays;        /* World::hit calls = ray segments (common.rs:268) */
  uint64_t samples;     /* pixel samples traced (width*height*spp of this shard) */
  float    kernel_ms;   /* device time of the render kernel, CUDA events */
  float    total_ms;    /* wall time of the call, copies included */
  uint32_t launches;    /* kernels launched */
  uint32_t grid;        /* CTAs of the persistent launch */
  uint32_t smem_bytes;  /* primitive-list bytes staged per CTA */
  uint32_t resident;    /* 1: primitive list lives in shared memory */
  uint32_t block;       /* threads per CTA */
  uint32_t devices;     /* GPUs that rendered this frame */
  uint32_t peer_gather; /* 1: shards stored their tiles straight into device 0's frame (NVLink peer stores) */
  uint32_t filtered;    /* 1: the exact kernel put its conservative FMA filter in front of the sphere tests */
  uint32_t sample_items;/* 1: work items were single samples; a second kernel summed them in order */
  uint32_t culled;      /* 1: the CULL kernels ran (RT_OPT_GROUP_CULL) */
  uint32_t passes_fused;/* progressive passes traced by ONE persistent launch (0 or 1: a plain frame) */
  uint32_t stolen_slots;/* pixel slots this call's GPU(s) took from other GPUs' shards (work stealing) */
  uint32_t paths_per_lane; /* 2: the FILTER kernels ran with two paths per lane (one sphere load serves two rays) */
  uint32_t reserved;
} RtRenderStats;

/* One shard's block for cross-GPU work stealing (rt_shard_block_bytes bytes of device memory owned by
 * the GPU that renders shard `shard_index`; mapped into the other processes with rt_ipc_open, or plain
 * peer access inside one process). */
typedef struct RtPeerQueue {
  void    *block;
  uint32_t shard_index;
  uint32_t reserved;
} RtPeerQueue;

/* common.rs:289-294 `Options`, extended.  Zero-initialise, then set struct_size. */
typedef struct RtRenderOptions {
  uint32_t struct_size;        /* sizeof(RtRenderOptions) */
  int32_t  samples_per_pixel;  /* common.rs:290 */
  int32_t  max_ray_bounces;    /* common.rs:291 */
  uint32_t seed;               /* 0 -> 2547549 (random.rs:9) */
  uint32_t flags;              /* RT_OPT_* */
  int32_t  sample_begin;       /* index of the first sample of this pass */
  int32_t  resolve_spp;        /* divisor of the resolve; 0 -> sample_begin + samples_per_pixel */
  int32_t  device;             /* CUDA ordinal; -1 -> current device */
  uint32_t tile_rows;          /* row-tile height of the shard decomposition; 0 -> 16 */
  uint32_t shard_index;        /* this call renders tiles shard_index, +shard_count, ... */
  uint32_t shard_count;        /* 0 -> 1 */
  uint32_t n_devices;          /* render_with_options only: > 1 -> this one process renders the frame on
                                  devices 0..n-1 (row tiles d, d+N, ...; tiles are stored straight into
                                  device 0's frame over NVLink).  0 -> environment RT_GPUS, else 1 */
  RtRenderStats *stats;        /* optional out */
  /* --- ABI version 2 (callers built against version 1 pass a smaller struct_size; these then read as 0) --- */
  uint32_t passes;             /* 0 or 1: one pass.  k > 1: samples_per_pixel is traced as k progressive passes of
                                  samples_per_pixel/k, the float4 sums going through device memory in between —
                                  all inside ONE persistent launch (no drain between passes).  The frame equals the
                                  single-pass frame bit for bit (common.rs:338-340 adds the samples in order). */
  uint32_t n_peer_queues;      /* rt_render_device, shard_count > 1, RT_OPT_FULL_FRAME_OUT: cross-GPU work stealing. */
  const RtPeerQueue *peer_queues; /* The blocks of ALL shard_count shards (this shard's own included), in the order
                                  in which the others are raided once this shard's own queue is empty. */
} RtRenderOptions;

/* Threading: like the reference (lib.rs is single-threaded, its callers block in render()), every render call of a
 * process is serialised by one internal mutex, whatever device it targets; calls from several threads are safe and
 * produce the frames they would produce alone.  The caller's current CUDA device is left as it was. */

/* Thread-local text of the last failure of any call in this library ("" if none). */
const char *rt_last_error(void);
uint32_t    rt_abi_version(void);
/* Number of CUDA devices visible (0 when there is none: every render call then fails). */
int         rt_device_count(void);

/* Destructors the reference lacks (lib.rs:42-45 leaks the handle). */
void rt_free_world(struct Rust_WorldHandle *handle);
void rt_free_camera(struct Rust_Camera *camera);

/* lib.rs:49-57 with the hard-coded Options::new(16, 8, None, true) replaced by `options`.
 * Same framebuffer contract as render(). */
struct Rust_CFramebuffer render_with_options(struct Rust_CFramebuffer framebuffer,
                                             const struct Rust_WorldHandle *handle,
                                             const RtRenderOptions *options);

/* Progressive frame for interactive callers (GameView.swift re-renders on every key press and
 * idles in between): every call adds options->samples_per_pixel samples to what earlier calls
 * accumulated for the same world, camera, size, seed, depth and kernel, keeps the float sums in
 * device memory, and writes the resolved frame; any change of those (camera moved, window
 * resized, world edited) starts over.  k calls of n spp produce exactly the bits of one call of
 * k*n spp.  *total_spp_out (optional) receives the samples per pixel in the frame. */
struct Rust_CFramebuffer rt_render_progressive(struct Rust_CFramebuffer framebuffer,
                                               const struct Rust_WorldHandle *handle,
                                               const RtRenderOptions *options, int32_t *total_spp_out);
void rt_progressive_reset(const struct Rust_WorldHandle *handle);

/* Device-resident variant for multi-GPU plumbing and benchmarks.  device_pixels: RGBA8 in
 * device memory — the full width*height frame when shard_count <= 1, otherwise this shard's
 * tiles packed back to back (rt_shard_pixel_count pixels).  device_accum: optional float4
 * sums, same indexing.  stream: a cudaStream_t, or NULL for the library's own stream
 * (then the call returns after the kernel has finished).  With a stream the call returns as soon as the work is
 * enqueued — unless the render needs the library's per-device scratch (sample-item scheduling of heavy scenes, fused
 * passes without a caller accumulator), which every launch on the device shares: then it returns after the kernel has
 * finished, so that renders in flight on different streams of one device never share scratch.  Returns 0 on success. */
int rt_render_device(const struct Rust_WorldHandle *handle, const RtRenderOptions *options,
                     size_t width, size_t height, void *device_pixels, void *device_accum,
                     void *stream);
/* First-hit buffers (depth, position, normal, albedo and primitive id of every pixel's camera ray): the auxiliary
 * outputs of a renderer, e.g. picking, segmentation masks, or the guide buffers of a denoiser.  Every pointer is device
 * memory of the target device or NULL (that buffer is not written); all float buffers are row-major, top row first,
 * like the RGBA8 frame:
 *   depth    float [H][W]     HitRecord.t (common.rs:237-258); +inf on a miss
 *   position float [H][W][3]  Ray::at(t) (common.rs:20); 0 on a miss
 *   normal   float [H][W][3]  spheres normalize((pos - c)/r) (common.rs:95), triangles the stored normal, not
 *                             face-forwarded (:165, :188); 0 on a miss
 *   albedo   float [H][W][3]  the material's colour (Dielectric: 1, 1, 1); on a miss the sky colour of the ray
 *                             (common.rs:276-281)
 *   prim     int32 [H][W]     sphere i -> i, triangle j -> (number of spheres) + j, in list order; -1 on a miss
 * Set struct_size = sizeof(RtAovBuffers) and reserved = 0. */
typedef struct RtAovBuffers {
  uint32_t struct_size;
  uint32_t reserved;
  float   *depth, *position, *normal, *albedo;
  int32_t *prim;
} RtAovBuffers;

/* World::hit of ONE camera ray per pixel — the ray render_with_options traces for sample options->sample_begin of that
 * pixel (same jitter draws, or (0.5, 0.5) with RT_OPT_FIXED_JITTER) — written to `buffers`, bit for bit what the
 * reference's HitRecord holds (exact arithmetic).  A caller can average calls with sample_begin = 0..k-1.
 * Reads seed, sample_begin, device, stats and the flags RT_OPT_FIXED_JITTER and RT_OPT_GROUP_CULL (same buffers,
 * fewer sphere tests).  Ignores samples_per_pixel, max_ray_bounces, resolve_spp, tile_rows, RT_OPT_PIXEL_ITEMS and
 * RT_OPT_SAMPLE_ITEMS, so a caller can pass its render options unchanged.  Fails (non-zero, rt_last_error), before any
 * device work and without touching the buffers, on RT_OPT_FAST_MATH, RT_OPT_ACCUM_IN / _OUT, RT_OPT_NO_RESOLVE,
 * RT_OPT_RESOLVE_EACH_PASS, RT_OPT_FULL_FRAME_OUT, RT_OPT_ROW_GATHER, RT_OPT_NO_STEAL, shard_count > 1, n_devices > 1,
 * passes > 1, peer queues, all buffers NULL, a frame smaller than 1x1 or wider / taller than 2^30 - 1, and a buffer
 * that is not device memory of the target device.  stream: a cudaStream_t, or NULL for the library's own stream (then
 * the call returns after the buffers are written); with a stream the call returns once the kernel is enqueued (unless
 * options->stats asks for the kernel time).  Stats: rays = samples = width*height, launches = 1.  Returns 0 on success. */
int rt_render_aov_device(const struct Rust_WorldHandle *handle, const RtRenderOptions *options,
                         size_t width, size_t height, const RtAovBuffers *buffers, void *stream);

/* Denoiser options.  Zero-initialise, set struct_size = sizeof(RtDenoiseOptions); a field left at 0 takes its default:
 *   iterations    1..10, default RT_DENOISE_DEFAULT_ITERATIONS (the a-trous steps are 1, 2, 4, ... 2^(iterations-1))
 *   sigma_color   finite, > 0: edge-stopping scale of the demodulated colour (default RT_DENOISE_DEFAULT_SIGMA_COLOR)
 *   sigma_normal  finite, > 0: of the normal difference (default RT_DENOISE_DEFAULT_SIGMA_NORMAL)
 *   sigma_plane   finite, > 0: of the distance of a neighbour's position to the pixel's tangent plane, in scene units
 *                 (default RT_DENOISE_DEFAULT_SIGMA_PLANE)
 *   device        CUDA device ordinal, -1 = the current device
 *   stats         optional out: kernel_ms, total_ms, launches (1 + iterations), grid and block; rays = samples = 0 */
#define RT_DENOISE_DEFAULT_ITERATIONS 5u
#define RT_DENOISE_DEFAULT_SIGMA_COLOR 1.0f
#define RT_DENOISE_DEFAULT_SIGMA_NORMAL 0.25f
#define RT_DENOISE_DEFAULT_SIGMA_PLANE 0.02f
typedef struct RtDenoiseOptions {
  uint32_t       struct_size;
  uint32_t       iterations;
  float          sigma_color, sigma_normal, sigma_plane;
  int32_t        device;
  RtRenderStats *stats;
} RtDenoiseOptions;

/* Edge-avoiding a-trous wavelet filter (Dammertz et al., HPG 2010) of a W x H frame's colour sums, guided by its
 * first-hit buffers; the result is bit for bit the same on every B200 and equals the CPU restatement of DESIGN.md §12.
 *   accum   float4 [H][W] colour sums, as rt_render_device writes them with RT_OPT_ACCUM_OUT (shard_count <= 1)
 *   spp     >= 1: the mean is m = sum * (1.0f / spp), alpha included (resolve's reciprocal-multiply)
 *   guides  normal, position, albedo and prim of rt_render_aov_device, all required (depth is ignored, may be NULL).
 *           A pixel with prim < 0 is a miss: never filtered, never a neighbour; its output is m.  Render the guides
 *           with RT_OPT_FIXED_JITTER and sample_begin = 0 to take them at pixel centres.
 * A hit pixel's colour is divided by a' = max(albedo, 2^-10) per channel, filtered `iterations` times with 5x5 taps at
 * steps 1, 2, 4, ... (edge-stopping weights (1 + u/16)^-16 of the colour, normal and plane-distance terms), and
 * multiplied by a' again; its alpha is m's, unfiltered.  Outputs, each optional but not both NULL, row-major, top row
 * first like the RGBA8 frame:
 *   device_pixels  RGBA8 [H][W]: the colour output resolved like a 1-spp frame (sqrt gamma, x255.999, `as u8`), so at a
 *                  miss pixel it equals rt_render_device's RGBA8 of the same sums
 *   device_color   float4 [H][W]: (filtered rgb * a', m.a) at a hit, m at a miss
 * Every pointer is device memory of the target device.  Fails (non-zero, rt_last_error), before any device work and
 * without touching the outputs, on NULL options or a wrong struct_size, iterations > 10, a sigma that is negative, NaN
 * or inf, spp < 1, a NULL accum, guides or required guide, both outputs NULL, a frame smaller than 1x1 or wider /
 * taller than 2^30 - 1, a buffer that is not device memory of the target device, and an output whose bytes overlap an
 * input's (or the other output's).  The call uses per-device scratch (64 bytes per pixel, kept between calls), so it
 * returns after the outputs are written, also with a caller's stream: stream is a cudaStream_t the work is ordered
 * on (after the caller's earlier work on it), or NULL for the library's own stream.  Returns 0 on success. */
int rt_denoise_device(const RtDenoiseOptions *options, size_t width, size_t height, const void *accum, int32_t spp,
                      const RtAovBuffers *guides, void *device_pixels, void *device_color, void *stream);

/* Ray queries: "what does this ray hit?" for rays the caller builds (picking at any point, line of sight, shadow rays
 * towards a light, baking).  Ray i is World::hit(Ray{o, d}, 0.001, t_max) (common.rs:237-258) of
 *   RtRay { float origin[3]; float t_max; float direction[3]; float reserved; }   (32 bytes, two float4; reserved ignored)
 * with these semantics, shared by the kernel and the CPU reference:
 *   1. Domain, checked per ray on the device.  A ray is valid when none of the seven floats is NaN, origin and
 *      direction are finite, |origin.c| <= 2^40 for every component, and s = (dx*dx + dy*dy) + dz*dz (float32, unfused,
 *      left to right) lies in [2^-100, 2^100]; t_max may be +-inf.  An invalid ray gets prim -2, depth NaN and 0 in
 *      position, normal and albedo: a bad ray never fails the call.
 *   2. d = the direction normalised as NVec3::new (maths.rs:111-118), the camera ray's own normalisation: the
 *      un-normalised camera vector ((llc + u*horizontal) + v*vertical) - origin gives exactly the camera ray.
 *   3. Closest hit with t_min = 0.001: a sphere hit counts when t < t_max (common.rs:88-92, strict), a triangle hit when
 *      t <= t_max (:142, inclusive); t_max = +inf is World::hit of the renderer's rays.
 *   4. Record, RtAovBuffers with arrays of n elements (ray i -> element i), each pointer optional:
 *        depth    float [n]     t; +inf on a miss
 *        position float [n][3]  Ray::at(t); 0 on a miss
 *        normal   float [n][3]  spheres normalize((pos - c)/r), triangles the stored normal (not face-forwarded); 0 on a miss
 *        albedo   float [n][3]  the material's colour (Dielectric 1, 1, 1); on a miss the sky colour of d
 *        prim     int32 [n]     sphere i -> i, triangle j -> (number of spheres) + j; -1 on a miss, -2 for an invalid ray
 *      With t_max = +inf and the camera vector of a pixel (fixed jitter) the record equals rt_render_aov_device's for
 *      that pixel, bit for bit. */
typedef struct RtRay {
  float origin[3];
  float t_max;
  float direction[3];
  float reserved;
} RtRay;

/* Options of rt_trace_rays_device.  Zero-initialise and set struct_size = sizeof(RtRayQueryOptions).
 *   flags   0 or RT_OPT_GROUP_CULL (same records, fewer sphere tests on large worlds); any other flag is rejected
 *   device  CUDA device ordinal, -1 = the current device
 *   stats   optional out: kernel_ms, total_ms, rays = samples = n, launches = 1, grid, block, smem_bytes, resident,
 *           filtered and culled */
typedef struct RtRayQueryOptions {
  uint32_t       struct_size;
  uint32_t       flags;
  int32_t        device;
  uint32_t       reserved;
  RtRenderStats *stats;
} RtRayQueryOptions;

/* The records of n rays (semantics above) into `hits`.  `rays` and every non-NULL pointer of `hits` are device memory of
 * the target device; `rays` is 16-byte aligned.  Fails (non-zero, rt_last_error), before any device work and without
 * touching the outputs, on a NULL handle, NULL options or a wrong struct_size, a flag other than RT_OPT_GROUP_CULL
 * (RT_OPT_FAST_MATH included), n == 0 or n > 2^31 - 1, a NULL or misaligned ray buffer, NULL hits or all of its
 * pointers NULL, a buffer that is not device memory of the target device, and an output whose bytes overlap the rays
 * or another output.  stream: a cudaStream_t, or NULL for the library's own stream (the call then returns after the
 * outputs are written).  That stream is non-blocking: it does not wait for work the caller enqueued on the legacy
 * default stream, so a caller that wrote the rays there passes cudaStreamLegacy (or synchronises first).  With a stream
 * the call returns once the kernel is enqueued, unless options->stats asks for the kernel time.  Uses no per-device
 * scratch.  Returns 0 on success. */
int rt_trace_rays_device(const struct Rust_WorldHandle *handle, const RtRayQueryOptions *options, size_t n,
                         const RtRay *rays, const RtAovBuffers *hits, void *stream);

/* Occlusion queries: "does anything lie on this segment?" for rays the caller builds (shadow rays towards a light, line
 * of sight, collision tests).  Ray i is an RtRay, checked and normalised exactly as in rt_trace_rays_device (items 1
 * and 2 above), and its answer is one byte:
 *   2  the ray is invalid (outside the domain of item 1); an invalid ray never fails the call
 *   1  World::hit(Ray{o, d}, 0.001, t_max) (common.rs:237-258) returns a hit
 *   0  it returns none
 * i.e. prim >= 0 ? 1 : prim == -1 ? 0 : 2 with the prim rt_trace_rays_device writes for the same ray.  World::hit
 * returns a hit exactly when some sphere's t = (root1 > 0.001 ? root1 : root2) satisfies 0.001 < t < t_max, or some
 * triangle's t passes its tests with the window [0.001, t_max] and t < +inf.  Each condition depends on one primitive,
 * so the walk stops at the first primitive that passes and the answer does not depend on the visiting order.
 * options: those of rt_trace_rays_device (flags 0 or RT_OPT_GROUP_CULL, device, stats with rays = samples = n,
 * launches = 1).  `rays` and `occluded` (n bytes) are device memory of the target device; `rays` is 16-byte aligned.
 * Fails (non-zero, rt_last_error), before any device work and without touching `occluded`, on a NULL handle, NULL
 * options or a wrong struct_size, a flag other than RT_OPT_GROUP_CULL, n == 0 or n > 2^31 - 1, a NULL or misaligned
 * ray buffer, a NULL `occluded`, memory that is not on the target device, and `occluded` overlapping the rays' 32*n
 * bytes.  stream: as for rt_trace_rays_device (NULL: the library's non-blocking stream, and the call returns when
 * `occluded` is written).  Uses no per-device scratch.  Returns 0 on success. */
int rt_occluded_rays_device(const struct Rust_WorldHandle *handle, const RtRayQueryOptions *options, size_t n,
                            const RtRay *rays, uint8_t *occluded, void *stream);

size_t rt_shard_pixel_count(size_t width, size_t height, uint32_t tile_rows,
                            uint32_t shard_index, uint32_t shard_count);

/* Cameras (camera.rs:21-69).  Each replaces handle->camera, freeing the old one.
 * Return 0 on success, non-zero where the reference asserts (camera.rs:50,:62). */
int rt_set_camera_at(struct Rust_WorldHandle *handle, const float origin[3], float aspect_ratio);
int rt_set_camera_vertical_fov(struct Rust_WorldHandle *handle, const float origin[3],
                               float vertical_fov_radians, float aspect_ratio);
int rt_set_camera_look_at(struct Rust_WorldHandle *handle, const float origin[3],
                          const float look_at[3], const float up[3],
                          float vertical_fov_radians, float aspect_ratio);
/* Install a camera verbatim: origin, lower_left_corner, horizontal, vertical (camera.rs:8-15)
 * as 12 floats — for callers that build the Camera with the crate's own constructors. */
int rt_set_camera_raw(struct Rust_WorldHandle *handle, const float camera12[12]);
/* origin, lower_left_corner, horizontal, vertical (camera.rs:8-15) as 12 floats. */
void  rt_get_camera(const struct Rust_Camera *camera, float out12[12]);
float rt_camera_aspect_ratio(const struct Rust_Camera *camera);   /* camera.rs:70-72 */

/* Scene construction without the text parser (World::new, common.rs:233-235; the only way
 * to reach MaterialType::Emission, which parser.rs cannot produce). */
struct Rust_WorldHandle *rt_world_new(const float camera_origin[3], float aspect_ratio);
int rt_world_add_sphere(struct Rust_WorldHandle *handle, const float center[3], float radius,
                        uint32_t material, const float color[3], float param);
int rt_world_add_triangle(struct Rust_WorldHandle *handle, const float v0[3], const float v1[3],
                          const float v2[3], uint32_t material, const float color[3], float param);
size_t rt_world_sphere_count(const struct Rust_WorldHandle *handle);
size_t rt_world_triangle_count(const struct Rust_WorldHandle *handle);
/* Read back primitive `index` in list (= hit-test) order.  out9: center[3], radius,
 * material type (as float), color[3], param.  out18: v0[3], v1[3], v2[3], stored normal[3],
 * material type, color[3], param, 0.  Return 0 on success. */
int rt_world_get_sphere(const struct Rust_WorldHandle *handle, size_t index, float out9[9]);
int rt_world_get_triangle(const struct Rust_WorldHandle *handle, size_t index, float out18[18]);

/* load_world with opt-in grammar extensions (load_world itself accepts exactly the reference's
 * grammar and rejects everything the reference rejects).  RT_PARSE_EMISSION: also accept
 * `material NAME : Emission color r g b;` — MaterialType::Emission exists (materials.rs:11) but
 * parser.rs:171-174 cannot produce it. */
#define RT_PARSE_EMISSION 0x1u
struct Rust_WorldHandle *rt_load_world_ext(const char *source, uint32_t extensions);

/* The inverse of load_world: the world (with its camera as `camera origin .. aspect ..`) in the
 * grammar of parser.rs:326-335, every float as its exact decimal expansion, so that
 * load_world(text) reproduces the primitives bit for bit.  Materials of type Emission are written
 * as `Emission color r g b` (read back with rt_load_world_ext + RT_PARSE_EMISSION).  Returns the size
 * needed including the terminating NUL (call with buffer = NULL to query); 0 on failure. */
size_t rt_world_to_text(const struct Rust_WorldHandle *handle, char *buffer, size_t capacity);

/* image.rs:59-81: ASCII PPM (P3), and a binary P6 variant.  Return 0 on success. */
int rt_write_image(struct Rust_CFramebuffer framebuffer, const char *path);
int rt_write_image_p6(struct Rust_CFramebuffer framebuffer, const char *path);

/* Pinned host frame buffers: render() DMA's straight into them. */
struct Rust_ColorU8 *rt_alloc_pixels(size_t width, size_t height);
void                 rt_free_pixels(struct Rust_ColorU8 *pixels);

/* Multi-process frame gather without a collective: rank 0 allocates the frame with
 * rt_device_alloc and exports it (CUDA IPC, 64-byte handle); every other rank opens it and
 * passes the mapped pointer as `device_pixels` of rt_render_device with RT_OPT_FULL_FRAME_OUT,
 * so its render kernel stores its tiles straight into rank 0's memory over NVLink.
 * rt_copy_to_host enqueues the final D2H on `stream`.  Pointers are NULL / results non-zero on
 * failure (rt_last_error). */
void *rt_device_alloc(size_t bytes);
/* Shard blocks (work stealing + fused passes across GPUs): size for a width x height frame, and the one-time
 * initialisation by the owner ("queue empty") before anybody may be given the block. */
size_t rt_shard_block_bytes(size_t width, size_t height);
int    rt_shard_block_init(void *block);
void  rt_device_free(void *device_ptr);
int   rt_ipc_export(const void *device_ptr, unsigned char handle_out[64]);
void *rt_ipc_open(const unsigned char handle[64]);
int   rt_ipc_close(void *mapped_ptr);
int   rt_copy_to_host(void *host_dst, const void *device_src, size_t bytes, void *stream);

/* FFMA-chain microbenchmark: measured FP32 peak of `device` in TFLOP/s (the roofline
 * denominator of the render kernel).  Negative on failure. */
double rt_measure_fp32_peak(int device);

/* GPU self-test: the exact kernel's shared-reciprocal divide (three numerators, one divisor)
 * against the compiler's IEEE divide on `operand_sets` pseudo-random operand sets.  Returns
 * the number of sets whose quotients differ in any bit (0 expected), negative on failure. */
long long rt_selftest_division(int device, unsigned long long operand_sets, uint32_t seed);
/* GPU self-test: the exact kernel's range-guarded square root (the compiler's own correctly rounded sequence without
 * its per-call range branch) against sqrtf on EVERY float bit pattern.  Returns the number of patterns whose bits
 * differ or whose range predicate is wrong (0 expected), negative on failure. */
long long rt_selftest_sqrt(int device);

#ifdef __cplusplus
}
#endif
#endif /* RAYTRACER_B200_H */
