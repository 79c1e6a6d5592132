// rt_capi.cpp — the C ABI (include/raytracer.h + include/raytracer_b200.h) over the C++
// host layer.  No exception crosses this boundary: failures set a thread-local error string.
#include "../../include/raytracer_b200.h"
#include "rt_host.hpp"

#include <cstddef>
#include <cstdlib>
#include <cstring>
#include <exception>
#include <stdexcept>
#include <string>

// The opaque ABI types are the C++ host objects.
// State of the progressive frame of rt_render_progressive (lives with the world).
struct Progressive {
    void*      d_accum = nullptr;      // float4 sums, device memory
    size_t     cap_px  = 0;
    int        device  = -1;
    size_t     width = 0, height = 0;
    rt::Camera camera{};
    uint32_t   seed = 0, flags = 0;
    int32_t    depth = 0;
    int32_t    done  = 0;              // samples per pixel accumulated so far
};
struct Rust_World  { std::unique_ptr<rt::World> world; Progressive progressive; };
struct Rust_Camera { rt::Camera camera; };

namespace {

thread_local std::string g_error;

void set_error(const std::string& s) { g_error = s; }
void clear_error() { g_error.clear(); }

// RT_GPUS=N lets an unchanged caller of render() (GameView.swift, examples/c_raytracer.rs) use N GPUs.
int env_devices()
{
    const char* e = std::getenv("RT_GPUS");
    if (!e || !*e) return 0;
    int n = std::atoi(e);
    return n > 0 ? n : 0;
}

rt::Options to_options(const RtRenderOptions* o)
{
    rt::Options r;
    if (!o) {                                        // render(): Options::new(16, 8, None, true), lib.rs:51
        r.samples_per_pixel = 16; r.max_ray_bounces = 8;
        // an unchanged caller of render() can still ask for the deterministic mode (fixed sub-pixel offset)
        const char* det = std::getenv("RT_DETERMINISTIC");
        r.fixed_jitter = det && *det && *det != '0';
        return r;
    }
    RtRenderOptions c;
    std::memset(&c, 0, sizeof c);
    std::memcpy(&c, o, o->struct_size && o->struct_size < sizeof c ? o->struct_size : sizeof c);
    r.samples_per_pixel = c.samples_per_pixel;
    r.max_ray_bounces   = c.max_ray_bounces;
    r.seed              = c.seed ? c.seed : 2547549u;
    r.fixed_jitter      = (c.flags & RT_OPT_FIXED_JITTER) != 0;
    r.fast_math         = (c.flags & RT_OPT_FAST_MATH) != 0;
    r.accum_in          = (c.flags & RT_OPT_ACCUM_IN) != 0;
    r.accum_out         = (c.flags & RT_OPT_ACCUM_OUT) != 0;
    r.no_resolve        = (c.flags & RT_OPT_NO_RESOLVE) != 0;
    r.full_frame_out    = (c.flags & RT_OPT_FULL_FRAME_OUT) != 0;
    r.group_cull        = (c.flags & RT_OPT_GROUP_CULL) != 0;
    r.n_devices         = (int32_t)c.n_devices;
    r.sample_items      = (c.flags & RT_OPT_SAMPLE_ITEMS) ? 1 : (c.flags & RT_OPT_PIXEL_ITEMS) ? 0 : -1;
    r.sample_begin      = c.sample_begin;
    r.resolve_spp       = c.resolve_spp;
    r.device            = c.device;
    r.tile_rows         = c.tile_rows ? c.tile_rows : 16u;
    r.shard_index       = c.shard_index;
    r.shard_count       = c.shard_count ? c.shard_count : 1u;
    r.passes            = c.passes > 1u ? (int32_t)c.passes : 1;
    r.resolve_each_pass = (c.flags & RT_OPT_RESOLVE_EACH_PASS) != 0;
    static_assert(sizeof(RtPeerQueue) == sizeof(rt::PeerQueue), "RtPeerQueue mirrors rt::PeerQueue");
    r.peer_queues       = reinterpret_cast<const rt::PeerQueue*>(c.peer_queues);
    r.n_peer_queues     = c.peer_queues ? c.n_peer_queues : 0u;
    r.no_steal          = (c.flags & RT_OPT_NO_STEAL) != 0;
    r.row_gather        = (c.flags & RT_OPT_ROW_GATHER) != 0;
    return r;
}

// A caller built against ABI version 1 passes the shorter RtRenderOptions and owns the shorter RtRenderStats:
// only the version-1 fields are written for it.
constexpr size_t kOptionsV1 = offsetof(RtRenderOptions, stats) + sizeof(RtRenderStats*);
RtRenderStats* stats_of(const RtRenderOptions* o) { return (o && o->struct_size >= kOptionsV1) ? o->stats : nullptr; }
bool           is_v2(const RtRenderOptions* o) { return o && o->struct_size >= sizeof(RtRenderOptions); }

void export_stats(const rt::RenderStats& s, RtRenderStats* out, bool v2)
{
    out->rays = s.rays; out->samples = s.samples; out->kernel_ms = s.kernel_ms; out->total_ms = s.total_ms;
    out->launches = s.launches; out->grid = s.grid; out->smem_bytes = s.smem_bytes; out->resident = s.resident;
    out->block = s.block; out->devices = s.devices; out->peer_gather = s.peer_gather; out->filtered = s.filtered;
    out->sample_items = s.sample_items; out->culled = s.culled;
    if (v2) { out->passes_fused = s.passes_fused; out->stolen_slots = s.stolen_slots; out->paths_per_lane = s.paths_per_lane; out->reserved = 0; }
}

template <class F>
int guarded(F&& f)
{
    clear_error();
    try { f(); return 0; }
    catch (const std::exception& e) { set_error(e.what()); }
    catch (...) { set_error("unknown error"); }
    return 1;
}

rt::Material make_material(uint32_t type, const float color[3], float param)
{
    rt::Material m;
    m.type = (RtMaterialType)type;
    m.r = color ? color[0] : 1.f; m.g = color ? color[1] : 1.f; m.b = color ? color[2] : 1.f;
    m.param = param;
    return m;
}

void replace_camera(Rust_WorldHandle* h, const rt::Camera& c)
{
    delete h->camera;
    h->camera = new Rust_Camera{c};
}

}   // namespace

extern "C" {

const char* rt_last_error(void) { return g_error.c_str(); }
uint32_t    rt_abi_version(void) { return RT_B200_ABI_VERSION; }
int         rt_device_count(void) { return rt::device_count(); }

static Rust_WorldHandle* load_world_impl(const char* source, bool allow_emission)
{
    clear_error();
    if (!source) { set_error("load_world: source is NULL"); return nullptr; }
    try {
        rt::ParseResult r = rt::parse_input(source, std::strlen(source), allow_emission);
        if (r.error != rt::ParseError::Ok) {
            set_error(std::string("load_world: ParseError: ") + rt::parse_error_name(r.error));
            return nullptr;
        }
        auto* h   = new Rust_WorldHandle;
        h->world  = new Rust_World{std::move(r.world), Progressive{}};
        h->camera = new Rust_Camera{r.camera};
        return h;
    } catch (const std::exception& e) {
        set_error(e.what());
        return nullptr;
    }
}

Rust_WorldHandle* load_world(const char* source) { return load_world_impl(source, false); }
Rust_WorldHandle* rt_load_world_ext(const char* source, uint32_t extensions)
{
    return load_world_impl(source, (extensions & RT_PARSE_EMISSION) != 0);
}

Rust_Camera* move_camera_position(Rust_Camera* camera, float x, float y, float z)
{
    clear_error();
    if (!camera) { set_error("move_camera_position: camera is NULL"); return nullptr; }
    auto* moved = new Rust_Camera{camera->camera.moved(x, y, z)};
    delete camera;   // Box<Camera> taken by value (lib.rs:60)
    return moved;
}

Rust_CFramebuffer render_with_options(Rust_CFramebuffer fb, const Rust_WorldHandle* handle,
                                      const RtRenderOptions* options)
{
    guarded([&] {
        if (!handle || !handle->world || !handle->camera) throw std::runtime_error("render: NULL world handle");
        if (!fb.pixels) throw std::runtime_error("render: framebuffer.pixels is NULL");
        rt::Options     o = to_options(options);
        rt::RenderStats st;
        RtRenderStats*  out_stats = stats_of(options);
        if (out_stats) o.stats = &st;
        const int n_dev = o.n_devices > 0 ? o.n_devices : env_devices();
        if (n_dev > 1 && o.shard_count <= 1)
            rt::ray_trace_multi(*handle->world->world, handle->camera->camera, fb.width, fb.height, o,
                                reinterpret_cast<rt::ColorU8*>(fb.pixels), n_dev);
        else if (rt::is_device_memory(fb.pixels))      // a caller that keeps its frame on the GPU (e.g. for display)
            rt::ray_trace_into(*handle->world->world, handle->camera->camera, fb.width, fb.height, o, nullptr,
                               fb.pixels, nullptr, nullptr);
        else
            rt::ray_trace_into(*handle->world->world, handle->camera->camera, fb.width, fb.height, o,
                               reinterpret_cast<rt::ColorU8*>(fb.pixels), nullptr, nullptr, nullptr);
        if (out_stats) export_stats(st, out_stats, is_v2(options));
    });
    return fb;
}

// SURVEY.md 8f-2: the interactive caller (GameView.swift re-renders on every key press, and sits
// idle in between).  Every call adds options->samples_per_pixel samples to the frame accumulated
// so far for the same world, camera, size, seed and depth — the sums stay in device memory, the
// sample indices continue where the last call stopped, so k calls of n spp give exactly the
// bits of one call of k*n spp — and starts over when any of those changed (camera moved,
// window resized, world edited).
Rust_CFramebuffer rt_render_progressive(Rust_CFramebuffer fb, const Rust_WorldHandle* handle,
                                        const RtRenderOptions* options, int32_t* total_spp_out)
{
    if (total_spp_out) *total_spp_out = 0;
    guarded([&] {
        if (!handle || !handle->world || !handle->camera) throw std::runtime_error("rt_render_progressive: NULL world handle");
        if (!fb.pixels) throw std::runtime_error("rt_render_progressive: framebuffer.pixels is NULL");
        rt::Options  o = to_options(options);
        Progressive& p = handle->world->progressive;
        if (o.samples_per_pixel < 1) throw std::runtime_error("rt_render_progressive: samples_per_pixel must be >= 1");
        if (o.shard_count > 1 || o.n_devices > 1) throw std::runtime_error("rt_render_progressive: single device only");
        const uint32_t key_flags = (o.fixed_jitter ? 1u : 0u) | (o.fast_math ? 2u : 0u);
        const bool same = p.d_accum && p.width == fb.width && p.height == fb.height && p.seed == o.seed &&
                          p.depth == o.max_ray_bounces && p.flags == key_flags && p.device == o.device &&
                          std::memcmp(&p.camera.d, &handle->camera->camera.d, sizeof p.camera.d) == 0;
        if (!same) {
            const size_t px = fb.width * fb.height;
            if (p.cap_px < px || p.device != o.device) {
                if (p.d_accum) rt::device_free(p.d_accum);
                p.d_accum = nullptr; p.cap_px = 0;
                p.d_accum = rt::device_alloc(px * 4 * sizeof(float), o.device);   // on the device that renders
                p.cap_px  = px;
            }
            p.width = fb.width; p.height = fb.height; p.seed = o.seed; p.depth = o.max_ray_bounces;
            p.flags = key_flags; p.device = o.device; p.camera = handle->camera->camera; p.done = 0;
        }
        rt::RenderStats st;
        RtRenderStats*  out_stats = stats_of(options);
        if (out_stats) o.stats = &st;
        o.sample_begin = p.done;
        o.resolve_spp  = p.done + o.samples_per_pixel;
        o.accum_in     = p.done > 0;
        o.accum_out    = true;
        o.no_resolve   = false;
        rt::ray_trace_into(*handle->world->world, handle->camera->camera, fb.width, fb.height, o,
                           reinterpret_cast<rt::ColorU8*>(fb.pixels), nullptr, p.d_accum, nullptr);
        p.done += o.samples_per_pixel;
        if (total_spp_out) *total_spp_out = p.done;
        if (out_stats) export_stats(st, out_stats, is_v2(options));
    });
    return fb;
}

void rt_progressive_reset(const Rust_WorldHandle* handle)
{
    if (handle && handle->world) handle->world->progressive.done = 0, handle->world->progressive.width = 0;
}

Rust_CFramebuffer render(Rust_CFramebuffer fb, const Rust_WorldHandle* handle)
{
    return render_with_options(fb, handle, nullptr);   // Options::new(16, 8, None, true), lib.rs:51
}

int rt_render_device(const Rust_WorldHandle* handle, const RtRenderOptions* options, size_t width, size_t height,
                     void* device_pixels, void* device_accum, void* stream)
{
    return guarded([&] {
        if (!handle || !handle->world || !handle->camera) throw std::runtime_error("rt_render_device: NULL world handle");
        rt::Options     o = to_options(options);
        rt::RenderStats st;
        RtRenderStats*  out_stats = stats_of(options);
        if (out_stats) o.stats = &st;
        if (!device_pixels && !o.no_resolve) throw std::runtime_error("rt_render_device: device_pixels is NULL");
        rt::ray_trace_into(*handle->world->world, handle->camera->camera, width, height, o, nullptr, device_pixels,
                           device_accum, stream);
        if (out_stats) export_stats(st, out_stats, is_v2(options));
    });
}

int rt_render_aov_device(const Rust_WorldHandle* handle, const RtRenderOptions* options, size_t width, size_t height,
                         const RtAovBuffers* buffers, void* stream)
{
    return guarded([&] {
        if (!handle || !handle->world || !handle->camera) throw std::runtime_error("rt_render_aov_device: NULL world handle");
        if (!buffers) throw std::runtime_error("rt_render_aov_device: buffers is NULL");
        RtAovBuffers b;
        std::memset(&b, 0, sizeof b);
        std::memcpy(&b, buffers, buffers->struct_size && buffers->struct_size < sizeof b ? buffers->struct_size : sizeof b);
        rt::Options     o = to_options(options);
        rt::RenderStats st;
        RtRenderStats*  out_stats = stats_of(options);
        if (out_stats) o.stats = &st;
        rt::AovBuffers ab;
        ab.depth = b.depth; ab.position = b.position; ab.normal = b.normal; ab.albedo = b.albedo; ab.prim = b.prim;
        rt::render_aov(*handle->world->world, handle->camera->camera, width, height, o, ab, stream);
        if (out_stats) export_stats(st, out_stats, is_v2(options));
    });
}

int rt_denoise_device(const RtDenoiseOptions* options, size_t width, size_t height, const void* accum, int32_t spp,
                      const RtAovBuffers* guides, void* device_pixels, void* device_color, void* stream)
{
    return guarded([&] {
        if (!options) throw std::runtime_error("rt_denoise_device: options is NULL");
        if (options->struct_size != sizeof(RtDenoiseOptions))
            throw std::runtime_error("rt_denoise_device: options->struct_size must be sizeof(RtDenoiseOptions)");
        if (!guides) throw std::runtime_error("rt_denoise_device: guides is NULL");
        RtAovBuffers g;
        std::memset(&g, 0, sizeof g);
        std::memcpy(&g, guides, guides->struct_size && guides->struct_size < sizeof g ? guides->struct_size : sizeof g);
        rt::DenoiseOptions o;
        o.iterations   = options->iterations;
        o.sigma_color  = options->sigma_color;
        o.sigma_normal = options->sigma_normal;
        o.sigma_plane  = options->sigma_plane;
        o.device       = options->device;
        rt::RenderStats st;
        if (options->stats) o.stats = &st;
        rt::DenoiseBuffers b;
        b.accum = accum; b.normal = g.normal; b.position = g.position; b.albedo = g.albedo; b.prim = g.prim;
        b.pixels = device_pixels; b.color = device_color;
        rt::denoise(o, width, height, spp, b, stream);
        if (options->stats) export_stats(st, options->stats, true);
    });
}

int rt_temporal_accumulate_device(const RtTemporalOptions* options, size_t width, size_t height, const void* accum,
                                  int32_t spp, const RtAovBuffers* guides, const float camera12[12],
                                  const RtTemporalHistory* history, void* color_out, float* length_out,
                                  void* device_pixels, void* stream)
{
    return guarded([&] {
        if (!options) throw std::runtime_error("rt_temporal_accumulate_device: options is NULL");
        if (options->struct_size != sizeof(RtTemporalOptions))
            throw std::runtime_error("rt_temporal_accumulate_device: options->struct_size must be sizeof(RtTemporalOptions)");
        if (!guides) throw std::runtime_error("rt_temporal_accumulate_device: guides is NULL");
        if (history && history->struct_size != sizeof(RtTemporalHistory))
            throw std::runtime_error("rt_temporal_accumulate_device: history->struct_size must be sizeof(RtTemporalHistory)");
        auto aov = [](const RtAovBuffers* in) {
            RtAovBuffers g;
            std::memset(&g, 0, sizeof g);
            if (in) std::memcpy(&g, in, in->struct_size && in->struct_size < sizeof g ? in->struct_size : sizeof g);
            return g;
        };
        const RtAovBuffers g = aov(guides);
        rt::TemporalOptions o;
        o.max_history = options->max_history;
        o.normal_cos  = options->normal_cos;
        o.plane_tol   = options->plane_tol;
        o.device      = options->device;
        rt::RenderStats st;
        if (options->stats) o.stats = &st;
        rt::TemporalBuffers b;
        b.accum = accum; b.position = g.position; b.normal = g.normal; b.prim = g.prim; b.camera = camera12;
        b.history = history != nullptr;
        if (history) {
            const RtAovBuffers pg = aov(history->guides);
            b.prev_camera = history->camera12;
            b.prev_position = pg.position; b.prev_normal = pg.normal; b.prev_prim = pg.prim;
            b.prev_color = history->color; b.prev_length = history->length;
        }
        b.color = color_out; b.length = length_out; b.pixels = device_pixels;
        rt::temporal(o, width, height, spp, b, stream);
        if (options->stats) export_stats(st, options->stats, true);
    });
}

int rt_svgf_device(const RtSvgfOptions* options, size_t width, size_t height, const void* accum, int32_t spp,
                   const RtAovBuffers* guides, const float camera12[12], const RtSvgfHistory* history, void* illum_out,
                   void* moments_out, float* length_out, void* device_pixels, void* device_color, void* stream)
{
    return guarded([&] {
        if (!options) throw std::runtime_error("rt_svgf_device: options is NULL");
        if (options->struct_size != sizeof(RtSvgfOptions))
            throw std::runtime_error("rt_svgf_device: options->struct_size must be sizeof(RtSvgfOptions)");
        if (!guides) throw std::runtime_error("rt_svgf_device: guides is NULL");
        if (history && history->struct_size != sizeof(RtSvgfHistory))
            throw std::runtime_error("rt_svgf_device: history->struct_size must be sizeof(RtSvgfHistory)");
        auto aov = [](const RtAovBuffers* in) {
            RtAovBuffers g;
            std::memset(&g, 0, sizeof g);
            if (in) std::memcpy(&g, in, in->struct_size && in->struct_size < sizeof g ? in->struct_size : sizeof g);
            return g;
        };
        const RtAovBuffers g = aov(guides);
        rt::SvgfOptions o;
        o.iterations      = options->iterations;
        o.max_history     = options->max_history;
        o.normal_cos      = options->normal_cos;
        o.plane_tol       = options->plane_tol;
        o.sigma_luminance = options->sigma_luminance;
        o.sigma_normal    = options->sigma_normal;
        o.sigma_plane     = options->sigma_plane;
        o.device          = options->device;
        rt::RenderStats st;
        if (options->stats) o.stats = &st;
        rt::SvgfBuffers b;
        b.accum = accum; b.position = g.position; b.normal = g.normal; b.albedo = g.albedo; b.prim = g.prim;
        b.camera = camera12;
        b.history = history != nullptr;
        if (history) {
            const RtAovBuffers pg = aov(history->guides);
            b.prev_camera = history->camera12;
            b.prev_position = pg.position; b.prev_normal = pg.normal; b.prev_prim = pg.prim;
            b.prev_illum = history->illum; b.prev_moments = history->moments; b.prev_length = history->length;
        }
        b.illum = illum_out; b.moments = moments_out; b.length = length_out;
        b.pixels = device_pixels; b.color = device_color;
        rt::svgf(o, width, height, spp, b, stream);
        if (options->stats) export_stats(st, options->stats, true);
    });
}

// The options of the two ray calls (rt_trace_rays_device, rt_occluded_rays_device), checked on the host; `call` prefixes
// every rejection.
static rt::RayQueryOptions ray_query_options(const char* call, const Rust_WorldHandle* handle,
                                             const RtRayQueryOptions* options, rt::RenderStats* st)
{
    const std::string c(call);
    if (!handle || !handle->world) throw std::runtime_error(c + ": NULL world handle");
    if (!options) throw std::runtime_error(c + ": options is NULL");
    if (options->struct_size != sizeof(RtRayQueryOptions))
        throw std::runtime_error(c + ": options->struct_size must be sizeof(RtRayQueryOptions)");
    if (options->flags & ~RT_OPT_GROUP_CULL)
        throw std::runtime_error(c + ": only RT_OPT_GROUP_CULL is supported in flags (RT_OPT_FAST_MATH "
                                     "and the render flags are not)");
    rt::RayQueryOptions o;
    o.group_cull = (options->flags & RT_OPT_GROUP_CULL) != 0;
    o.device     = options->device;
    if (options->stats) o.stats = st;
    return o;
}

int rt_trace_rays_device(const Rust_WorldHandle* handle, const RtRayQueryOptions* options, size_t n, const RtRay* rays,
                         const RtAovBuffers* hits, void* stream)
{
    return guarded([&] {
        rt::RenderStats           st;
        const rt::RayQueryOptions o = ray_query_options("rt_trace_rays_device", handle, options, &st);
        if (!hits) throw std::runtime_error("rt_trace_rays_device: hits is NULL");
        RtAovBuffers b;
        std::memset(&b, 0, sizeof b);
        std::memcpy(&b, hits, hits->struct_size && hits->struct_size < sizeof b ? hits->struct_size : sizeof b);
        rt::AovBuffers ab;
        ab.depth = b.depth; ab.position = b.position; ab.normal = b.normal; ab.albedo = b.albedo; ab.prim = b.prim;
        rt::trace_rays(*handle->world->world, o, n, rays, ab, stream);
        if (options->stats) export_stats(st, options->stats, true);
    });
}

int rt_occluded_rays_device(const Rust_WorldHandle* handle, const RtRayQueryOptions* options, size_t n,
                            const RtRay* rays, uint8_t* occluded, void* stream)
{
    return guarded([&] {
        rt::RenderStats           st;
        const rt::RayQueryOptions o = ray_query_options("rt_occluded_rays_device", handle, options, &st);
        rt::occluded_rays(*handle->world->world, o, n, rays, occluded, stream);
        if (options->stats) export_stats(st, options->stats, true);
    });
}

size_t rt_shard_pixel_count(size_t width, size_t height, uint32_t tile_rows, uint32_t shard_index, uint32_t shard_count)
{
    if (!tile_rows) tile_rows = 16;
    if (!shard_count) shard_count = 1;
    if (shard_count == 1) return width * height;
    return (size_t)rt::shard_tile_count((uint32_t)height, tile_rows, shard_index, shard_count) * tile_rows * width;
}

void rt_free_world(Rust_WorldHandle* h)
{
    if (!h) return;
    if (h->world && h->world->progressive.d_accum) rt::device_free(h->world->progressive.d_accum);
    delete h->world;
    delete h->camera;
    delete h;
}
void rt_free_camera(Rust_Camera* c) { delete c; }

int rt_set_camera_at(Rust_WorldHandle* h, const float origin[3], float aspect)
{
    return guarded([&] {
        if (!h) throw std::runtime_error("NULL world handle");
        replace_camera(h, rt::Camera::new_at(RtVec3{origin[0], origin[1], origin[2]}, aspect));
    });
}
int rt_set_camera_vertical_fov(Rust_WorldHandle* h, const float origin[3], float vfov, float aspect)
{
    return guarded([&] {
        if (!h) throw std::runtime_error("NULL world handle");
        replace_camera(h, rt::Camera::new_with_vertical_fov(RtVec3{origin[0], origin[1], origin[2]}, vfov, aspect));
    });
}
int rt_set_camera_look_at(Rust_WorldHandle* h, const float origin[3], const float look_at[3], const float up[3],
                          float vfov, float aspect)
{
    return guarded([&] {
        if (!h) throw std::runtime_error("NULL world handle");
        rt::Camera  c;
        std::string err;
        if (!rt::Camera::new_look_at(RtVec3{origin[0], origin[1], origin[2]}, RtVec3{look_at[0], look_at[1], look_at[2]},
                                     RtVec3{up[0], up[1], up[2]}, vfov, aspect, &c, &err))
            throw std::runtime_error(err);
        replace_camera(h, c);
    });
}
int rt_set_camera_raw(Rust_WorldHandle* h, const float camera12[12])
{
    return guarded([&] {
        if (!h || !camera12) throw std::runtime_error("NULL world handle or camera");
        rt::Camera c;
        std::memcpy(&c.d, camera12, 12 * sizeof(float));
        replace_camera(h, c);
    });
}
void rt_get_camera(const Rust_Camera* camera, float out12[12])
{
    if (!camera) return;
    std::memcpy(out12, &camera->camera.d, 12 * sizeof(float));
}
float rt_camera_aspect_ratio(const Rust_Camera* camera) { return camera ? camera->camera.aspect_ratio() : 0.f; }

Rust_WorldHandle* rt_world_new(const float origin[3], float aspect)
{
    clear_error();
    auto* h   = new Rust_WorldHandle;
    h->world  = new Rust_World{rt::World::make({}, {}), Progressive{}};
    h->camera = new Rust_Camera{rt::Camera::new_at(origin ? RtVec3{origin[0], origin[1], origin[2]} : RtVec3{0, 0, 0}, aspect)};
    return h;
}
int rt_world_add_sphere(Rust_WorldHandle* h, const float center[3], float radius, uint32_t material,
                        const float color[3], float param)
{
    return guarded([&] {
        if (!h || !h->world) throw std::runtime_error("NULL world handle");
        if (material > RT_MATERIAL_EMISSION) throw std::runtime_error("unknown material type");
        h->world->world->spheres.push_back(rt::Sphere{RtVec3{center[0], center[1], center[2]}, radius,
                                                      make_material(material, color, param)});
        h->world->world->invalidate_device();
        rt_progressive_reset(h);
    });
}
int rt_world_add_triangle(Rust_WorldHandle* h, const float v0[3], const float v1[3], const float v2[3],
                          uint32_t material, const float color[3], float param)
{
    return guarded([&] {
        if (!h || !h->world) throw std::runtime_error("NULL world handle");
        if (material > RT_MATERIAL_EMISSION) throw std::runtime_error("unknown material type");
        h->world->world->triangles.push_back(rt::Triangle::make(RtVec3{v0[0], v0[1], v0[2]}, RtVec3{v1[0], v1[1], v1[2]},
                                                                RtVec3{v2[0], v2[1], v2[2]},
                                                                make_material(material, color, param)));
        h->world->world->invalidate_device();
        rt_progressive_reset(h);
    });
}
size_t rt_world_sphere_count(const Rust_WorldHandle* h) { return (h && h->world) ? h->world->world->spheres.size() : 0; }
size_t rt_world_triangle_count(const Rust_WorldHandle* h) { return (h && h->world) ? h->world->world->triangles.size() : 0; }

int rt_world_get_sphere(const Rust_WorldHandle* h, size_t i, float out[9])
{
    if (!h || !h->world || i >= h->world->world->spheres.size()) return 1;
    const rt::Sphere& s = h->world->world->spheres[i];
    const float v[9] = {s.center.x, s.center.y, s.center.z, s.radius, (float)s.material.type,
                        s.material.r, s.material.g, s.material.b, s.material.param};
    std::memcpy(out, v, sizeof v);
    return 0;
}
int rt_world_get_triangle(const Rust_WorldHandle* h, size_t i, float out[18])
{
    if (!h || !h->world || i >= h->world->world->triangles.size()) return 1;
    const rt::Triangle& t = h->world->world->triangles[i];
    const float v[18] = {t.v0.x, t.v0.y, t.v0.z, t.v1.x, t.v1.y, t.v1.z, t.v2.x, t.v2.y, t.v2.z,
                         t.normal.x, t.normal.y, t.normal.z, (float)t.material.type,
                         t.material.r, t.material.g, t.material.b, t.material.param, 0.f};
    std::memcpy(out, v, sizeof v);
    return 0;
}

size_t rt_world_to_text(const Rust_WorldHandle* h, char* buffer, size_t capacity)
{
    size_t need = 0;
    guarded([&] {
        if (!h || !h->world || !h->camera) throw std::runtime_error("NULL world handle");
        const std::string s = rt::world_to_text(*h->world->world, h->camera->camera);
        need = s.size() + 1;
        if (buffer && capacity >= need) std::memcpy(buffer, s.c_str(), need);
    });
    return need;
}

static int write_any(Rust_CFramebuffer fb, const char* path, bool p6)
{
    return guarded([&] {
        if (!fb.pixels) throw std::runtime_error("framebuffer.pixels is NULL");
        const rt::ColorU8* px = reinterpret_cast<const rt::ColorU8*>(fb.pixels);
        if (!(p6 ? rt::write_image_p6(px, fb.width, fb.height, path) : rt::write_image(px, fb.width, fb.height, path)))
            throw std::runtime_error("cannot write image");
    });
}
int rt_write_image(Rust_CFramebuffer fb, const char* path) { return write_any(fb, path, false); }
int rt_write_image_p6(Rust_CFramebuffer fb, const char* path) { return write_any(fb, path, true); }

Rust_ColorU8* rt_alloc_pixels(size_t width, size_t height)
{
    clear_error();
    void* p = rt::alloc_pinned(width * height * 4);
    if (!p) set_error("rt_alloc_pixels: pinned allocation failed (no CUDA device?)");
    return static_cast<Rust_ColorU8*>(p);
}
void rt_free_pixels(Rust_ColorU8* pixels) { rt::free_pinned(pixels); }

void* rt_device_alloc(size_t bytes)
{
    void* p = nullptr;
    guarded([&] { p = rt::device_alloc(bytes); });
    return p;
}
void rt_device_free(void* p) { rt::device_free(p); }
size_t rt_shard_block_bytes(size_t width, size_t height) { return rt::shard_block_bytes(width, height); }
int    rt_shard_block_init(void* block) { return guarded([&] { rt::shard_block_init(block); }); }
int  rt_ipc_export(const void* device_ptr, unsigned char handle_out[64])
{
    return guarded([&] { rt::ipc_export(device_ptr, handle_out); });
}
void* rt_ipc_open(const unsigned char handle[64])
{
    void* p = nullptr;
    guarded([&] { p = rt::ipc_open(handle); });
    return p;
}
int rt_ipc_close(void* p) { return guarded([&] { rt::ipc_close(p); }); }
int rt_copy_to_host(void* host_dst, const void* device_src, size_t bytes, void* stream)
{
    return guarded([&] { rt::copy_to_host(host_dst, device_src, bytes, stream); });
}

double rt_measure_fp32_peak(int device)
{
    double v = -1.0;
    guarded([&] { v = rt::measure_fp32_peak_tflops(device, nullptr); });
    return v;
}

long long rt_selftest_division(int device, unsigned long long operand_sets, uint32_t seed)
{
    long long v = -1;
    guarded([&] { v = rt::selftest_division(device, operand_sets, seed); });
    return v;
}

long long rt_selftest_sqrt(int device)
{
    long long v = -1;
    guarded([&] { v = rt::selftest_sqrt(device); });
    return v;
}

}   // extern "C"
