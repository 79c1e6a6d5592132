// rt_host.hpp — C++ host layer above the CUDA kernels.
//
// The reference's host side is Rust; this image has no Rust toolchain, so the host layer is
// C++ that mirrors the crate's public API for the render path name for name:
//
//   reference (raytracer/src/...)                      here (namespace rt)
//   ---------------------------------------------------------------------------------
//   materials.rs:7-12   MaterialType                   Material
//   common.rs:54-58     Sphere                         Sphere
//   common.rs:101-123   Triangle, Triangle::new        Triangle, Triangle::make
//   common.rs:227-235   World, World::new              World, World::make
//   camera.rs:8-72      Camera, new_at, new_with_vertical_fov, new_look_at, aspect_ratio
//   common.rs:289-317   Options                        Options (+ seed / flags / sharding)
//   image.rs:9-36       Framebuffer                    Framebuffer
//   common.rs:320-361   ray_trace                      ray_trace           (runs on the GPU)
//   parser.rs:336-382   parse_input                    parse_input
//   image.rs:59-81      write_image                    write_image
//
// There is no CPU implementation of ray_trace in this library: without a CUDA device every
// render call fails with an error (never a silent fallback).
#pragma once
#include "rt_types.h"

#include <cstddef>
#include <cstdint>
#include <memory>
#include <string>
#include <vector>

namespace rt {

// materials.rs:7-12
struct Material {
    RtMaterialType type  = RT_MAT_DIFFUSE;
    float          r = 0.f, g = 0.f, b = 0.f;   // Color (alpha == 1, color.rs:21-23)
    float          param = 0.f;                 // Metal: fuzz, Dielectric: ir
    static Material Diffuse(float r, float g, float b) { return {RT_MAT_DIFFUSE, r, g, b, 0.f}; }
    static Material Metal(float r, float g, float b, float fuzz) { return {RT_MAT_METAL, r, g, b, fuzz}; }
    static Material Dielectric(float ir) { return {RT_MAT_DIELECTRIC, 1.f, 1.f, 1.f, ir}; }
    static Material Emission(float r, float g, float b) { return {RT_MAT_EMISSION, r, g, b, 0.f}; }
};

// common.rs:54-58
struct Sphere {
    RtVec3   center;
    float    radius;
    Material material;
};

// common.rs:101-107
struct Triangle {
    RtVec3   v0, v1, v2;
    RtVec3   normal;     // normalize((v1-v0) x (v2-v0)), common.rs:116-123
    Material material;
    static Triangle make(RtVec3 v0, RtVec3 v1, RtVec3 v2, const Material& m);
};

// camera.rs:8-15
struct Camera {
    RtCameraData d;
    static Camera new_at(RtVec3 origin, float aspect_ratio);                              // :21-33
    static Camera new_with_vertical_fov(RtVec3 origin, float vfov_radians, float aspect); // :34-48
    // :49-69.  Returns false (and sets *error) where the reference asserts.
    static bool new_look_at(RtVec3 origin, RtVec3 look_at, RtVec3 up, float vfov_radians, float aspect,
                            Camera* out, std::string* error);
    float  aspect_ratio() const { return d.horizontal.x / d.vertical.y; }                 // :70-72
    RtVec3 position() const { return d.origin; }                                          // :91-93
    Camera moved(float x, float y, float z) const;                                        // lib.rs:60-63
};

// image.rs:9-36 + color.rs:3-10
struct ColorU8 { uint8_t r, g, b, a; };
struct Framebuffer {
    size_t               width = 0, height = 0;
    std::vector<ColorU8> pixels;   // row-major, top row first
    Framebuffer() = default;
    Framebuffer(size_t w, size_t h) : width(w), height(h), pixels(w * h, ColorU8{0, 0, 0, 0}) {}
};

// Per-render statistics (additive; the reference reports nothing).
// One shard's block for cross-GPU work stealing: [work counter, 256 B][float4 sums, width*height].
struct PeerQueue { void* block; uint32_t shard_index; uint32_t reserved; };
size_t shard_block_bytes(size_t width, size_t height);
void   shard_block_init(void* block);        // marks the queue empty (call once after allocating, on the owner)

struct RenderStats {
    uint64_t rays       = 0;     // World::hit calls (ray segments)
    uint64_t samples    = 0;     // pixel samples traced
    float    kernel_ms  = 0.f;   // device time of the render kernel(s), CUDA events
    float    total_ms   = 0.f;   // wall time of the call including copies
    uint32_t launches   = 0;     // kernels launched by this call
    uint32_t grid       = 0;
    uint32_t smem_bytes = 0;
    uint32_t resident   = 0;     // 1: primitive list staged in shared memory
    uint32_t block      = 0;     // threads per CTA
    uint32_t devices    = 1;     // GPUs that rendered this frame
    uint32_t peer_gather = 0;    // 1: shards stored their tiles straight into device 0's frame (NVLink peer stores)
    uint32_t filtered   = 0;     // 1: exact kernel ran its conservative sphere filter (large sphere lists)
    uint32_t sample_items = 0;   // 1: work items were single samples (ordered sum by the resolve kernel)
    uint32_t culled     = 0;     // 1: the CULL kernels ran (group bounds in front of the filter)
    uint32_t passes_fused = 0;   // progressive passes traced by one persistent launch (0/1: a plain frame)
    uint32_t stolen_slots = 0;   // pixel slots this GPU took from other GPUs' shards (cross-GPU work stealing)
    uint32_t paths_per_lane = 1; // 2: every lane traced two paths and tested both rays against each sphere it loaded
};

// common.rs:289-294, extended.  The reference fields keep their names.
struct Options {
    int32_t  samples_per_pixel = 32;        // Options::default(), common.rs:309-316
    int32_t  max_ray_bounces   = 8;
    bool     positive_is_up    = true;      // stored, never read (as in the reference)
    // ---- additive ----
    uint32_t seed           = 2547549u;     // random.rs:9
    bool     fixed_jitter   = false;        // deterministic mode: sub-pixel offset (0.5, 0.5)
    bool     fast_math      = false;        // relaxed-arithmetic kernel (not bit-exact)
    int32_t  sample_begin   = 0;            // first sample index of this pass
    int32_t  resolve_spp    = 0;            // 0: sample_begin + samples_per_pixel
    int32_t  device         = -1;           // CUDA device ordinal, -1: current device
    uint32_t tile_rows      = 16;           // row-tile height of the shard decomposition
    uint32_t shard_index    = 0;            // this shard renders tiles shard_index, +shard_count, ...
    uint32_t shard_count    = 1;
    bool     accum_in       = false;        // continue from the float4 accumulator (progressive)
    bool     accum_out      = false;        // write the float4 accumulator back
    bool     no_resolve     = false;        // skip the RGBA8 pack (intermediate pass)
    bool     full_frame_out = false;        // sharded, but device_pixels/device_accum are FULL frames (e.g. a
                                            // peer-mapped frame on another GPU): tiles land at their frame offset
    int32_t  n_devices      = 0;            // > 1: one process drives devices 0..n-1 (ray_trace_multi)
    int32_t  sample_items   = -1;           // work-item granularity: -1 auto, 0 whole pixels, 1 single samples
    bool     group_cull     = false;        // opt-in: skip whole groups of spheres through bounding spheres (same
                                            // hits; a separately reported mode — it changes the work done)
    // Progressive passes: samples_per_pixel is traced as `passes` passes of samples_per_pixel/passes, the
    // float4 sums going through device memory between passes (k x n spp == k*n spp bit for bit).  All
    // passes run in ONE persistent launch (pass-major work queue, rt_types.h) unless the frame continues
    // an accumulator (accum_in) or uses sample items, where a single pass of the total is traced instead.
    int32_t  passes            = 1;
    bool     resolve_each_pass = false;     // fused passes: the RGBA8 frame is refreshed after every pass
    // Cross-GPU work stealing (shard_count > 1 with full_frame_out): the shard blocks (shard_block_bytes)
    // of ALL shards of the frame, this shard's own among them, each in its owner's device memory and
    // mapped here (peer access / CUDA IPC).  Order = the order in which the others are raided.
    const PeerQueue* peer_queues   = nullptr;
    uint32_t         n_peer_queues = 0;
    bool     no_steal       = false;        // peer_queues given, but every GPU traces only its own shard
    // device_pixels is a full frame in ANOTHER GPU's memory (peer access / CUDA IPC): render into a local, zeroed frame
    // with the same kernel and let a small second kernel move every pixel found there across as 16-byte vectors,
    // instead of one 4-byte store per pixel over NVLink ("row gather").  Needs full_frame_out and whole-pixel items.
    bool     row_gather     = false;
    RenderStats* stats      = nullptr;
};

struct DeviceScene;   // per-device packed scene (defined in rt_device.cu)

// common.rs:227-235.  Holds the primitives in list order and the lazily built device copies.
struct World {
    std::vector<Sphere>   spheres;
    std::vector<Triangle> triangles;     // the single Mesh of lib.rs:41 / main.rs:58-79
    World();
    ~World();
    World(const World&)            = delete;
    World& operator=(const World&) = delete;
    static std::unique_ptr<World> make(std::vector<Sphere> spheres, std::vector<Triangle> triangles);
    void invalidate_device();            // call after editing spheres/triangles
    // packed host copy of the scene blob (rt_types.h layout), built on demand
    struct Packed {
        std::vector<unsigned char> blob;
        size_t off_sph = 0, off_tri_plane = 0, off_sph_filter = 0, off_sph_r2 = 0, off_tri_cull = 0, off_tri_v = 0,
               off_info = 0, off_cull_bound = 0, off_cull_sph = 0, off_cull_r2 = 0, off_cull_orig = 0;
        uint32_t n_sph = 0, n_sph_pad = 0, n_tri = 0, n_tri_pad = 0, n_groups = 0;
        RtSceneView view(const unsigned char* base) const;
    };
    const Packed& packed() const;
    // internal
    mutable std::unique_ptr<Packed>                   packed_;
    mutable std::vector<std::unique_ptr<DeviceScene>> device_;
};

// parser.rs:10-17
enum class ParseError { Ok = 0, CouldntOpenFile, MissingCamera, WrongSyntax, DidntStartWith, NotAI32, NotAF32, InvalidUtf8 };
const char* parse_error_name(ParseError e);

struct ParseResult {
    ParseError             error = ParseError::Ok;
    Camera                 camera{};
    std::unique_ptr<World> world;
};
// parser.rs:336-382 (source need not be NUL-terminated here)
// allow_emission: also accept `material NAME : Emission color r g b;` (an extension; off = the reference's grammar)
ParseResult parse_input(const char* source, size_t length, bool allow_emission = false);

// The inverse of parse_input: `world` + a new_at camera in the reference's grammar, every float
// as its exact decimal expansion (parse_input(world_to_text(w)) reproduces w bit for bit).
std::string world_to_text(const World& world, const Camera& camera);

// First-hit buffers of render_aov: device memory of the target device, row-major, top row first; a null pointer
// means "not written".
struct AovBuffers {
    float*   depth    = nullptr;   // [H][W]
    float*   position = nullptr;   // [H][W][3]
    float*   normal   = nullptr;   // [H][W][3]
    float*   albedo   = nullptr;   // [H][W][3]
    int32_t* prim     = nullptr;   // [H][W]
};

// World::hit (common.rs:237-258) of the camera ray of sample options.sample_begin of every pixel — the ray
// ray_trace traces for that sample — written to `buffers` (exact arithmetic).  Reads seed, sample_begin, device,
// stats, fixed_jitter and group_cull; ignores samples_per_pixel, max_ray_bounces, resolve_spp, tile_rows and the
// scheduling options; rejects every other option.  stream: nullptr = the library's stream (returns when the
// buffers are written), else the call returns once the kernel is enqueued.  Throws std::runtime_error.
void render_aov(const World& world, const Camera& camera, size_t width, size_t height, const Options& options,
                const AovBuffers& buffers, void* stream);

// Ray queries (rt_ray_kernel): World::hit(Ray{o, normalize(direction)}, 0.001, t_max) of n caller-supplied rays
// (DESIGN.md §13).  `rays` holds n records {origin[3], t_max, direction[3], reserved} (RtRay), 16-byte aligned; the
// record of ray i goes to element i of the non-null buffers of `hits` (AovBuffers with arrays of length n).  Only
// group_cull of the options is read.  Rejects, before any device work and without touching the outputs: n == 0 or
// n > 2^31 - 1, a null or misaligned ray buffer, all outputs null, a buffer that is not device memory of the target
// device, and an output whose bytes overlap the rays or another output.  stream: nullptr = the library's stream
// (returns when the outputs are written), else the call returns once the kernel is enqueued (unless stats are asked
// for).  Throws std::runtime_error.
struct RayQueryOptions {
    bool         group_cull = false;
    int32_t      device     = -1;       // CUDA device ordinal, -1: current device
    RenderStats* stats      = nullptr;
};
void trace_rays(const World& world, const RayQueryOptions& options, size_t n, const void* rays, const AovBuffers& hits,
                void* stream);

// Occlusion queries (rt_occlusion_kernel): does World::hit(Ray{o, normalize(direction)}, 0.001, t_max) return a hit?
// (DESIGN.md §14).  The rays, options, stream and stats of trace_rays; occluded[i] = 1 (a hit), 0 (none) or 2 (an
// invalid ray).  Rejects what trace_rays rejects, with a null `occluded` for "all outputs null" and the n bytes of
// `occluded` as the one output.  Throws std::runtime_error.
void occluded_rays(const World& world, const RayQueryOptions& options, size_t n, const void* rays, uint8_t* occluded,
                   void* stream);

// Denoiser (rt_denoise.cu): a field left at 0 takes its default.  The defaults are chosen by the sigma sweep of
// scripts/denoise_bench.py (DESIGN.md §12) and repeated in include/raytracer_b200.h.
constexpr uint32_t kDenoiseDefaultIterations  = 5u;
constexpr uint32_t kDenoiseMaxIterations      = 10u;
constexpr float    kDenoiseDefaultSigmaColor  = 1.0f;
constexpr float    kDenoiseDefaultSigmaNormal = 0.25f;
constexpr float    kDenoiseDefaultSigmaPlane  = 0.02f;

struct DenoiseOptions {
    uint32_t     iterations   = 0;        // 1..10, 0: kDenoiseDefaultIterations
    float        sigma_color  = 0.f;      // finite, > 0; 0: the default
    float        sigma_normal = 0.f;
    float        sigma_plane  = 0.f;      // scene units
    int32_t      device       = -1;       // CUDA device ordinal, -1: current device
    RenderStats* stats        = nullptr;
};

// Device buffers of denoise, row-major, top row first.  accum, normal, position, albedo and prim are required; at
// least one of pixels / color.
struct DenoiseBuffers {
    const void*    accum    = nullptr;    // float4 [H][W] colour sums
    const float*   normal   = nullptr;    // [H][W][3]  first-hit guides (render_aov)
    const float*   position = nullptr;    // [H][W][3]
    const float*   albedo   = nullptr;    // [H][W][3]
    const int32_t* prim     = nullptr;    // [H][W]
    void*          pixels   = nullptr;    // RGBA8 [H][W] out
    void*          color    = nullptr;    // float4 [H][W] out
};

// Edge-avoiding a-trous filter of the mean colour sum / spp, guided by the first-hit buffers (DESIGN.md §12: bit for
// bit what tests/test_denoise.py's reference computes).  Uses per-device scratch, so the call is finished before it
// returns, also on a caller's stream.  stream: nullptr = the library's stream.  Throws std::runtime_error, before any
// device work and without touching the outputs when an argument is rejected.
void denoise(const DenoiseOptions& options, size_t width, size_t height, int32_t spp, const DenoiseBuffers& buffers,
             void* stream);

// Temporal accumulation (rt_temporal.cu): a field left at 0 takes its default.  The defaults are chosen by the sweep of
// scripts/temporal_bench.py (DESIGN.md §15) and repeated in include/raytracer_b200.h.
constexpr uint32_t kTemporalDefaultMaxHistory = 8u;
constexpr uint32_t kTemporalMaxMaxHistory     = 1u << 20;
constexpr float    kTemporalDefaultNormalCos  = 0.9f;
constexpr float    kTemporalDefaultPlaneTol   = 0.02f;

struct TemporalOptions {
    uint32_t     max_history = 0;         // 1..2^20, 0: kTemporalDefaultMaxHistory
    float        normal_cos  = 0.f;       // finite, in [-1, 1]; 0: the default
    float        plane_tol   = 0.f;       // finite, > 0, scene units; 0: the default
    int32_t      device      = -1;        // CUDA device ordinal, -1: current device
    RenderStats* stats       = nullptr;
};

// Device buffers of temporal, row-major, top row first.  The current frame's accum, position, normal, prim and camera
// are required, and so are color and length; with `history` every prev_* is required, without it they are not read.
struct TemporalBuffers {
    bool           history       = false;     // a previous frame is given
    const void*    accum         = nullptr;   // float4 [H][W] colour sums
    const float*   position      = nullptr;   // [H][W][3]  first-hit guides (render_aov)
    const float*   normal        = nullptr;   // [H][W][3]
    const int32_t* prim          = nullptr;   // [H][W]
    const float*   camera        = nullptr;   // 12 floats: origin, lower_left_corner, horizontal, vertical
    const float*   prev_camera   = nullptr;
    const float*   prev_position = nullptr;
    const float*   prev_normal   = nullptr;
    const int32_t* prev_prim     = nullptr;
    const void*    prev_color    = nullptr;   // float4 [H][W]: the previous call's color output
    const float*   prev_length   = nullptr;   // [H][W]: the previous call's length output
    void*          color         = nullptr;   // float4 [H][W] out
    float*         length        = nullptr;   // [H][W] out
    void*          pixels        = nullptr;   // RGBA8 [H][W] out, optional
};

// The colour sums / spp blended with the previous frame's colour history (DESIGN.md §15: bit for bit what
// tests/test_temporal.py's reference computes).  One kernel, no scratch: stream nullptr = the library's stream (returns
// when the outputs are written), else the call returns once the kernel is enqueued (unless stats are asked for).
// Throws std::runtime_error, before any device work and without touching the outputs when an argument is rejected.
void temporal(const TemporalOptions& options, size_t width, size_t height, int32_t spp, const TemporalBuffers& buffers,
              void* stream);

// Variance-guided filtering (rt_svgf.cu): a field left at 0 takes its default.  The defaults are chosen by the sweep of
// scripts/svgf_bench.py (DESIGN.md §16) and repeated in include/raytracer_b200.h.
constexpr uint32_t kSvgfDefaultIterations     = 5u;
constexpr uint32_t kSvgfDefaultMaxHistory     = 8u;
constexpr float    kSvgfDefaultNormalCos      = 0.9f;
constexpr float    kSvgfDefaultPlaneTol       = 0.02f;
constexpr float    kSvgfDefaultSigmaLuminance = 0.5f;
constexpr float    kSvgfDefaultSigmaNormal    = 0.25f;
constexpr float    kSvgfDefaultSigmaPlane     = 0.02f;

struct SvgfOptions {
    uint32_t     iterations      = 0;     // 1..10, 0: kSvgfDefaultIterations
    uint32_t     max_history     = 0;     // 1..2^20, 0: kSvgfDefaultMaxHistory
    float        normal_cos      = 0.f;   // finite, in [-1, 1]; 0: the default
    float        plane_tol       = 0.f;   // finite, > 0, scene units; 0: the default
    float        sigma_luminance = 0.f;   // finite, > 0; 0: the default
    float        sigma_normal    = 0.f;
    float        sigma_plane     = 0.f;   // scene units
    int32_t      device          = -1;    // CUDA device ordinal, -1: current device
    RenderStats* stats           = nullptr;
};

// Device buffers of svgf, row-major, top row first.  The current frame's accum, guides (position, normal, albedo,
// prim) and camera are required, and so are illum, moments and length; at least one of pixels / color.  With `history`
// every prev_* is required, without it they are not read.
struct SvgfBuffers {
    bool           history       = false;     // a previous frame is given
    const void*    accum         = nullptr;   // float4 [H][W] colour sums
    const float*   position      = nullptr;   // [H][W][3]  first-hit guides (render_aov)
    const float*   normal        = nullptr;   // [H][W][3]
    const float*   albedo        = nullptr;   // [H][W][3]
    const int32_t* prim          = nullptr;   // [H][W]
    const float*   camera        = nullptr;   // 12 floats: origin, lower_left_corner, horizontal, vertical
    const float*   prev_camera   = nullptr;
    const float*   prev_position = nullptr;
    const float*   prev_normal   = nullptr;
    const int32_t* prev_prim     = nullptr;
    const void*    prev_illum    = nullptr;   // float4 [H][W]: the previous call's illum output
    const void*    prev_moments  = nullptr;   // float2 [H][W]: its moments output
    const float*   prev_length   = nullptr;   // [H][W]: its length output
    void*          illum         = nullptr;   // float4 [H][W] out
    void*          moments       = nullptr;   // float2 [H][W] out
    float*         length        = nullptr;   // [H][W] out
    void*          pixels        = nullptr;   // RGBA8 [H][W] out
    void*          color         = nullptr;   // float4 [H][W] out
};

// Temporal accumulation of the demodulated colour and its luminance moments, a variance estimate per pixel, and the
// a-trous filter with that variance setting each pixel's colour weight (DESIGN.md §16: bit for bit what
// tests/test_svgf.py's reference computes).  Uses per-device scratch, so the call is finished before it returns, also
// on a caller's stream.  stream: nullptr = the library's stream.  Throws std::runtime_error, before any device work and
// without touching the outputs when an argument is rejected.
void svgf(const SvgfOptions& options, size_t width, size_t height, int32_t spp, const SvgfBuffers& buffers,
          void* stream);

// common.rs:320-361 on the GPU.  Renders into framebuffer.pixels and returns it.
// Throws std::runtime_error on any CUDA failure (no CPU fallback exists).
Framebuffer ray_trace(const World& world, const Camera& camera, Framebuffer framebuffer, Options& options);

// The same render with explicit destinations:
//  host_pixels   : width*height RGBA8 in host memory (pageable or pinned), or nullptr
//  device_pixels : RGBA8 in device memory (full frame, or this shard's tiles packed when
//                  shard_count > 1), or nullptr to use an internal buffer
//  device_accum  : optional float4 accumulator in device memory (progressive passes)
//  stream        : cudaStream_t (nullptr: the library's own stream, call is synchronous)
void ray_trace_into(const World& world, const Camera& camera, size_t width, size_t height,
                    const Options& options, ColorU8* host_pixels, void* device_pixels,
                    void* device_accum, void* stream);

// The same frame rendered by `n_devices` GPUs driven from this one process: device d renders
// row tiles d, d+N, ... and stores them straight into device 0's frame over NVLink peer
// mappings; device 0 sends the finished frame to host_pixels.
void ray_trace_multi(const World& world, const Camera& camera, size_t width, size_t height,
                     const Options& options, ColorU8* host_pixels, int n_devices);

// Number of rows / pixels shard `index` of `count` owns for an image of `height` rows.
uint32_t shard_tile_count(uint32_t height, uint32_t tile_rows, uint32_t index, uint32_t count);

// image.rs:59-81 (ASCII P3) and a binary P6 variant.  Return false on I/O failure.
bool write_image(const Framebuffer& fb, const char* path);
bool write_image_p6(const Framebuffer& fb, const char* path);
bool write_image(const ColorU8* pixels, size_t width, size_t height, const char* path);      // no copy of the frame
bool write_image_p6(const ColorU8* pixels, size_t width, size_t height, const char* path);

// Device utilities
int    device_count();
// FFMA-chain microbenchmark: measured FP32 peak of `device` in TFLOP/s (FMA = 2 flops).
double measure_fp32_peak_tflops(int device, float* sm_clock_mhz_out);
// GPU self-test of the shared-reciprocal divide against the compiler's IEEE divide on
// `operand_sets` pseudo-random operand sets; returns the number of mismatching sets.
long long selftest_division(int device, unsigned long long operand_sets, uint32_t seed);
// GPU self-test of the range-guarded square root (rt_trace.cuh sqrt_ranged) against sqrtf on every float bit
// pattern; returns the number of mismatching patterns.
long long selftest_sqrt(int device);
// Device memory that can be mapped into other processes (CUDA IPC): rank 0 owns the frame,
// the other ranks' kernels store their tiles into it.  All throw std::runtime_error on failure.
void* device_alloc(size_t bytes, int device = -1);   // -1: the current device
void  device_free(void* p);
void  ipc_export(const void* device_ptr, unsigned char handle_out[64]);
void* ipc_open(const unsigned char handle[64]);
void  ipc_close(void* p);
void  copy_to_host(void* host_dst, const void* device_src, size_t bytes, void* stream);
// Pinned host allocations for callers that want the frame DMA'd straight into their buffer.
bool  is_device_memory(const void* p);   // true for cudaMalloc'ed memory (a frame that should stay on the GPU)
void* alloc_pinned(size_t bytes);
void  free_pinned(void* p);

}   // namespace rt
