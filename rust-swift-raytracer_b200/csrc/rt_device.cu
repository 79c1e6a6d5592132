// rt_device.cu — device management and render orchestration (host side of the CUDA path).
//
//   World  --(pack, once)-->  scene blob  --(one H2D copy per device, once)-->  HBM
//   ray_trace_into():  [memset 16 B counters] -> ONE persistent render kernel -> [D2H frame]
//
// No CPU fallback: every failure becomes a std::runtime_error carrying the CUDA error text.
#include "rt_host.hpp"

#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <stdexcept>
#include <string>
#include <thread>
#include <tuple>
#include <vector>

namespace rt {

// defined in rt_kernels_exact.cu / rt_kernels_fast.cu
cudaError_t launch_render_exact(const RtFrameParams&, const RtSceneView&, int grid, size_t smem_limit, cudaStream_t);
cudaError_t launch_render_fast(const RtFrameParams&, const RtSceneView&, int grid, size_t smem_limit, cudaStream_t);
cudaError_t occupancy_exact(const RtSceneView& G, size_t smem_limit, bool cull, int* blocks_per_sm, int* block_size,
                            size_t* hot_bytes, int* resident, int* sph_mode);
cudaError_t occupancy_fast(const RtSceneView& G, size_t smem_limit, bool cull, int* blocks_per_sm, int* block_size,
                           size_t* hot_bytes, int* resident, int* sph_mode);
cudaError_t launch_resolve_samples_exact(const RtFrameParams&, cudaStream_t);
cudaError_t launch_aov_exact(const RtAovParams&, const RtSceneView&, bool cull, int grid, size_t smem_limit, cudaStream_t);
cudaError_t aov_occupancy_exact(const RtSceneView& G, size_t smem_limit, bool cull, int* blocks_per_sm, int* block_size,
                                size_t* hot_bytes, int* resident, int* sph_mode);
cudaError_t launch_rays_exact(const RtRayParams&, const RtSceneView&, bool cull, int grid, size_t smem_limit, cudaStream_t);
cudaError_t rays_occupancy_exact(const RtSceneView& G, size_t smem_limit, bool cull, int* blocks_per_sm, int* block_size,
                                 size_t* hot_bytes, int* resident, int* sph_mode);
cudaError_t launch_occlusion_exact(const RtOcclusionParams&, const RtSceneView&, bool cull, int grid, size_t smem_limit,
                                   cudaStream_t);
cudaError_t occlusion_occupancy_exact(const RtSceneView& G, size_t smem_limit, bool cull, int* blocks_per_sm,
                                      int* block_size, size_t* hot_bytes, int* resident, int* sph_mode);
cudaError_t launch_resolve_samples_fast(const RtFrameParams&, cudaStream_t);
cudaError_t launch_denoise(const RtDenoiseParams&, int num_sms, uint32_t* grid, uint32_t* block, cudaStream_t);   // rt_denoise.cu
cudaError_t launch_selftest_division(unsigned long long n_per_thread, uint32_t seed, int grid, int block,
                                     unsigned long long* d_mismatches, cudaStream_t);
cudaError_t launch_selftest_sqrt(int grid, int block, unsigned long long* d_mismatches, cudaStream_t);
cudaError_t launch_gather_rows(const uint32_t* local, uint32_t* remote, size_t n_pixels, int grid, cudaStream_t);
cudaError_t launch_ffma_peak(float* out, int iters, int grid, int block, cudaStream_t);
double      ffma_peak_flops_per_launch(int iters, int grid, int block);

namespace {

[[noreturn]] void fail(const char* what, cudaError_t e)
{
    throw std::runtime_error(std::string(what) + ": " + cudaGetErrorName(e) + " (" + cudaGetErrorString(e) + ")");
}
#define RT_CUDA(expr) do { cudaError_t e_ = (expr); if (e_ != cudaSuccess) fail(#expr, e_); } while (0)

constexpr int      kCounterSlots    = 64;
constexpr uint64_t kSampleBufferCap = (uint64_t)1 << 30;

struct CounterSlot {            // 16 B, zeroed by one memset per launch
    unsigned long long rays;
    unsigned int       work;
    unsigned int       stolen;
};

// Shard block (cross-GPU work stealing): the shard's work counter, alone in its first 256 bytes, then
// the float4 sums of the fused passes for the full frame.  Lives in its owner's device memory; the
// other GPUs reach it through peer access or a CUDA-IPC mapping.
constexpr size_t       kBlockHeader    = 256;
// layout of a shard block for a width x height frame: [header: the work counter][float4 sums, indexed like the frame]
struct BlockLayout { size_t off_accum, bytes; };
BlockLayout block_layout(size_t W, size_t H)
{
    BlockLayout b;
    b.off_accum = kBlockHeader;
    b.bytes     = b.off_accum + W * H * sizeof(RtFloat4);
    return b;
}
constexpr unsigned int kQueueExhausted = 0xC0000000u;   // any value >= every queue length (< 2^31)

struct DeviceContext {
    int          device   = -1;
    int          num_sms  = 0;
    size_t       smem_optin = 0;
    cudaStream_t stream   = nullptr;
    cudaEvent_t  ev0 = nullptr, ev1 = nullptr;
    std::vector<cudaEvent_t> ev_chunk;
    CounterSlot* d_slots  = nullptr;
    CounterSlot* h_slot   = nullptr;   // pinned
    int          next_slot = 0;
    uint32_t*    d_out    = nullptr;   size_t d_out_cap = 0;     // internal frame buffer (pixels)
    unsigned char* h_stage = nullptr;  size_t h_stage_cap = 0;   // pinned staging for pageable destinations
    RtFloat4*    d_samples = nullptr;  size_t d_samples_cap = 0; // per-sample colours of the sample-item mode
    RtFloat4*    d_accum = nullptr;    size_t d_accum_cap = 0;   // hand-over sums between sample-item chunks / fused passes
    unsigned char* d_block = nullptr;  size_t d_block_cap = 0;   // this device's shard block (ray_trace_multi)
    uint32_t*    d_local_frame = nullptr; size_t d_local_cap = 0;  // row gather: this shard's pixels before they cross NVLink
    unsigned int* d_tile_done = nullptr; unsigned int* h_tile_flags = nullptr; size_t tile_cap = 0;   // tile completion
    uint32_t     tile_epoch = 0;
    RtFloat4*    d_denoise = nullptr;  size_t d_denoise_cap = 0; // denoise: two colour frames + packed guides (float4s)
    struct Geometry { int per_sm = 0, block = 0, resident = 0, sph_mode = 0; size_t hot_bytes = 0; };
    std::map<std::tuple<uint32_t, uint32_t, uint32_t, int, int>, Geometry> occupancy;   // (Sp, Tp, groups, fast, cull) -> launch geometry
    std::map<std::tuple<uint32_t, uint32_t, uint32_t, int>, Geometry> aov_occupancy;    // (Sp, Tp, groups, cull) -> first-hit kernel
    std::map<std::tuple<uint32_t, uint32_t, uint32_t, int>, Geometry> ray_occupancy;    // (Sp, Tp, groups, cull) -> ray-query kernel
    std::map<std::tuple<uint32_t, uint32_t, uint32_t, int>, Geometry> occlusion_occupancy;   // likewise -> occlusion kernel
};

std::mutex                    g_mutex;          // one render at a time per process (lib.rs is single-threaded)
std::map<int, DeviceContext*> g_contexts;

DeviceContext& context_for(int device)
{
    auto it = g_contexts.find(device);
    if (it != g_contexts.end()) return *it->second;
    auto* c = new DeviceContext();
    c->device = device;
    RT_CUDA(cudaSetDevice(device));
    int v = 0;
    RT_CUDA(cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, device));
    c->num_sms = v;
    RT_CUDA(cudaDeviceGetAttribute(&v, cudaDevAttrMaxSharedMemoryPerBlockOptin, device));
    c->smem_optin = (size_t)v;
    RT_CUDA(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    RT_CUDA(cudaEventCreate(&c->ev0));
    RT_CUDA(cudaEventCreate(&c->ev1));
    RT_CUDA(cudaMalloc(&c->d_slots, kCounterSlots * sizeof(CounterSlot)));
    RT_CUDA(cudaMallocHost(&c->h_slot, sizeof(CounterSlot)));
    g_contexts[device] = c;
    return *c;
}

// Makes `device` current and restores the caller's current device when the scope ends.
struct DeviceGuard {
    int previous = -1;
    explicit DeviceGuard(int device)
    {
        if (cudaGetDevice(&previous) != cudaSuccess) { cudaGetLastError(); previous = -1; }
        RT_CUDA(cudaSetDevice(device));
    }
    ~DeviceGuard() { if (previous >= 0) cudaSetDevice(previous); }
    DeviceGuard(const DeviceGuard&)            = delete;
    DeviceGuard& operator=(const DeviceGuard&) = delete;
};

int resolve_device(int requested)
{
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0)
        throw std::runtime_error(std::string("no CUDA device available (this library has no CPU render path): ") +
                                 (e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0"));
    int dev = requested;
    if (dev < 0) RT_CUDA(cudaGetDevice(&dev));
    if (dev >= n) throw std::runtime_error("CUDA device ordinal out of range");
    return dev;
}

}   // namespace

// Per-device copy of the packed scene.
struct DeviceScene {
    int            device = -1;
    unsigned char* blob   = nullptr;
    size_t         bytes  = 0;
    RtSceneView    view{};
    ~DeviceScene()
    {
        if (blob) {
            int cur = -1;
            cudaGetDevice(&cur);
            cudaSetDevice(device);
            cudaFree(blob);
            if (cur >= 0) cudaSetDevice(cur);
        }
    }
};

World::World()  = default;
World::~World() = default;

void World::invalidate_device()
{
    std::lock_guard<std::mutex> lock(g_mutex);
    packed_.reset();
    device_.clear();
}

namespace {

// Scene upload (K1): one cudaMemcpy of the SoA blob, cached per (world, device).
const DeviceScene& device_scene(const World& w, DeviceContext& ctx)
{
    for (auto& s : w.device_)
        if (s->device == ctx.device) return *s;
    const World::Packed& p = w.packed();
    auto s    = std::make_unique<DeviceScene>();
    s->device = ctx.device;
    s->bytes  = p.blob.size();
    RT_CUDA(cudaMalloc(&s->blob, s->bytes));
    RT_CUDA(cudaMemcpyAsync(s->blob, p.blob.data(), s->bytes, cudaMemcpyHostToDevice, ctx.stream));
    RT_CUDA(cudaStreamSynchronize(ctx.stream));
    s->view = p.view(s->blob);
    w.device_.push_back(std::move(s));
    return *w.device_.back();
}

// Device-side address of a pinned (page-locked, mapped) host allocation, or nullptr.
void* mapped_device_pointer(const void* p)
{
    static const bool enabled = [] { const char* e = std::getenv("RT_ZERO_COPY"); return !(e && *e == '0'); }();
    if (!enabled) return nullptr;
    cudaPointerAttributes a;
    cudaError_t e = cudaPointerGetAttributes(&a, p);
    if (e != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return a.type == cudaMemoryTypeHost ? a.devicePointer : nullptr;
}

bool is_pinned_or_device_accessible(const void* p)
{
    cudaPointerAttributes a;
    cudaError_t e = cudaPointerGetAttributes(&a, p);
    if (e != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost || a.type == cudaMemoryTypeManaged;
}

}   // namespace

namespace {

// One shard's launch, enqueued on `stream` of ctx's device (which must be current).
struct ShardLaunch {
    uint32_t     n_tiles = 0;
    bool         compact = false;
    size_t       out_pixels = 0;
    int          grid = 0, block = 0;
    size_t       hot_bytes = 0, smem_limit = 0;
    bool         resident = false, filtered = false, culled = false, sample_items = false;
    uint32_t     launches = 0, passes_fused = 0, paths_per_lane = 1;
    bool         tile_flags = false;       // the kernel publishes per-tile completion flags (ctx.h_tile_flags, ctx.tile_epoch)
    bool         uses_scratch = false;     // the launch reads/writes per-device scratch (sample buffer, hand-over sums, frame)
    CounterSlot* slot = nullptr;
    uint32_t*    d_out = nullptr;
};

void validate_size(size_t width, size_t height)
{
    if (width < 1 || height < 1) throw std::runtime_error("framebuffer must be at least 1x1");
    if (width > 0x3fffffffu || height > 0x3fffffffu) throw std::runtime_error("framebuffer too large");
}

void validate(size_t width, size_t height, const Options& opt, const void* device_accum)
{
    validate_size(width, height);
    if (opt.tile_rows < 4 || (opt.tile_rows & 3u)) throw std::runtime_error("tile_rows must be a positive multiple of 4");
    if (opt.shard_count < 1 || opt.shard_index >= opt.shard_count) throw std::runtime_error("bad shard index/count");
    if ((opt.accum_in || opt.accum_out) && !device_accum && !opt.n_peer_queues)
        throw std::runtime_error("accumulator requested but device_accum is null");
    if (opt.passes > 1 && (opt.samples_per_pixel % opt.passes) != 0)
        throw std::runtime_error("samples_per_pixel must be a multiple of passes");
    if (opt.n_peer_queues) {
        if (opt.n_peer_queues > RT_MAX_QUEUES) throw std::runtime_error("too many peer queues");
        if (opt.n_peer_queues != opt.shard_count) throw std::runtime_error("peer_queues must list every shard of the frame");
        if (!opt.full_frame_out) throw std::runtime_error("work stealing needs a full-frame destination (RT_OPT_FULL_FRAME_OUT)");
        if (opt.accum_in || opt.accum_out || opt.no_resolve || device_accum)
            throw std::runtime_error("work stealing keeps its sums in the shard blocks: no caller accumulator");
    }
}

ShardLaunch enqueue_shard(DeviceContext& ctx, const DeviceScene& scene, const Camera& camera, uint32_t W, uint32_t H,
                          const Options& opt, uint32_t* d_out_in, void* device_accum, cudaStream_t stream, bool timed,
                          bool want_tile_flags = false)
{
    ShardLaunch L;
    L.n_tiles = shard_tile_count(H, opt.tile_rows, opt.shard_index, opt.shard_count);
    const uint64_t slots = (uint64_t)L.n_tiles * ((W + 7u) / 8u) * (opt.tile_rows / 4u) * 32u;
    L.compact    = opt.shard_count > 1 && !opt.full_frame_out;
    L.out_pixels = L.compact ? (size_t)L.n_tiles * opt.tile_rows * W : (size_t)W * H;

    L.d_out = d_out_in;
    if (!L.d_out && !opt.no_resolve) {
        if (ctx.d_out_cap < L.out_pixels) {
            if (ctx.d_out) RT_CUDA(cudaFree(ctx.d_out));
            ctx.d_out = nullptr; ctx.d_out_cap = 0;
            RT_CUDA(cudaMalloc(&ctx.d_out, L.out_pixels * sizeof(uint32_t)));
            ctx.d_out_cap = L.out_pixels;
        }
        L.d_out = ctx.d_out;
    }
    L.slot = ctx.d_slots + (ctx.next_slot++ % kCounterSlots);

    const bool trace = opt.samples_per_pixel > 0 && opt.max_ray_bounces > 0;

    RtFrameParams P{};
    P.camera       = camera.d;
    P.wm1          = (float)(W - 1u);      // `(width - 1) as f32`, common.rs:335
    P.hm1          = (float)(H - 1u);
    P.width        = W;
    P.height       = H;
    P.spp          = opt.samples_per_pixel;
    P.depth        = opt.max_ray_bounces;
    P.sample_begin = opt.sample_begin;
    P.resolve_spp  = opt.resolve_spp ? opt.resolve_spp : opt.sample_begin + opt.samples_per_pixel;
    P.seed         = opt.seed;
    P.flags        = (opt.fixed_jitter ? RT_FLAG_FIXED_JITTER : 0u) | (opt.accum_in ? RT_FLAG_ACCUM_IN : 0u) |
              (opt.accum_out ? RT_FLAG_ACCUM_OUT : 0u) | (opt.no_resolve ? RT_FLAG_NO_RESOLVE : 0u) |
              (L.compact ? RT_FLAG_COMPACT_OUT : 0u) | (opt.group_cull ? RT_FLAG_GROUP_CULL : 0u);
    P.tile_rows    = opt.tile_rows;
    P.div_subtiles_x       = rt_divisor((W + 7u) >> 3);
    P.div_chunks_per_strip = rt_divisor(((W + 7u) >> 3) * (opt.tile_rows >> 2));
    P.tile_first   = opt.shard_index;
    P.tile_stride  = opt.shard_count;
    P.n_tiles      = L.n_tiles;
    P.passes       = 1;
    P.one          = 1.0f;
    P.out          = L.d_out;
    P.accum        = static_cast<RtFloat4*>(device_accum);
    P.ray_counter  = &L.slot->rays;
    P.work_counter = &L.slot->work;
    P.steal_counter = &L.slot->stolen;

    // Work-item granularity.  A lane normally owns a whole pixel (all its samples, summed in
    // order in registers).  When the frame offers only a few pixels per lane and every ray
    // segment is expensive (large primitive lists), the drain at the end of the launch — lanes
    // idle while the last pixels finish — costs a large part of the run; then the work items
    // become single SAMPLES, their colours go to a buffer in HBM and a second kernel adds them
    // in sample order (same bits) and resolves.  Costs spp*32 B of HBM traffic per pixel, which
    // is why it is reserved for scenes whose segments cost thousands of instructions.
    int32_t chunk_spp = opt.samples_per_pixel;       // samples per launch in sample-item mode
    {
        const uint64_t lanes_max  = (uint64_t)ctx.num_sms * 2048u / 2u;          // paths in flight: 32 warps/SM at 64 registers
                                                                                 // (or 16 warps/SM carrying two paths per lane)
        const uint64_t pixels     = (uint64_t)L.n_tiles * opt.tile_rows * W;
        const uint64_t prims      = (uint64_t)scene.view.n_sph + scene.view.n_tri;
        const bool     want = opt.sample_items > 0 ||
                              (opt.sample_items < 0 && prims >= 512 && opt.samples_per_pixel >= 4 &&
                               pixels < 16u * lanes_max);
        L.sample_items = want && trace && L.n_tiles > 0;
        if (L.sample_items) {
            // the sample buffer is capped (1 GiB): more samples than fit are traced in several
            // launches that hand their sums on through the float4 accumulator
            const uint64_t per_sample = L.out_pixels * sizeof(RtFloat4);
            const uint64_t cap_spp    = std::max<uint64_t>(kSampleBufferCap / std::max<uint64_t>(per_sample, 1), 1);
            const uint64_t slot_spp   = std::max<uint64_t>(0x7fffff00ull / std::max<uint64_t>(slots, 1), 1) - 0;
            chunk_spp = (int32_t)std::min<uint64_t>({(uint64_t)opt.samples_per_pixel, cap_spp, slot_spp});
            const uint64_t buf_bytes = per_sample * (uint64_t)chunk_spp;
            if (ctx.d_samples_cap < buf_bytes) {
                RT_CUDA(cudaStreamSynchronize(stream));
                if (ctx.d_samples) RT_CUDA(cudaFree(ctx.d_samples));
                ctx.d_samples = nullptr; ctx.d_samples_cap = 0;
                RT_CUDA(cudaMalloc(&ctx.d_samples, buf_bytes));
                ctx.d_samples_cap = buf_bytes;
            }
            if (chunk_spp < opt.samples_per_pixel && !P.accum) {      // internal hand-over accumulator
                const size_t need = L.out_pixels * sizeof(RtFloat4);
                if (ctx.d_accum_cap < need) {
                    RT_CUDA(cudaStreamSynchronize(stream));
                    if (ctx.d_accum) RT_CUDA(cudaFree(ctx.d_accum));
                    ctx.d_accum = nullptr; ctx.d_accum_cap = 0;
                    RT_CUDA(cudaMalloc(&ctx.d_accum, need));
                    ctx.d_accum_cap = need;
                }
                P.accum = ctx.d_accum;
            }
            P.flags |= RT_FLAG_SAMPLE_ITEMS;
            P.samples       = ctx.d_samples;
            P.sample_stride = (uint32_t)L.out_pixels;
        }
    }

    // Cross-GPU work stealing and tile gather: the queue table of this launch, own shard first.
    const BlockLayout BL = block_layout(W, H);
    const bool     have_blocks = opt.n_peer_queues > 0 && !L.sample_items && trace;
    const bool     stealing    = have_blocks && opt.n_peer_queues > 1 && !opt.no_steal;
    unsigned char* own_block = nullptr;
    for (uint32_t i = 0; i < opt.n_peer_queues; ++i)
        if (opt.peer_queues[i].shard_index == opt.shard_index) own_block = static_cast<unsigned char*>(opt.peer_queues[i].block);
    if (opt.n_peer_queues && !own_block) throw std::runtime_error("peer_queues does not contain this shard's own block");
    auto queue_of = [&](unsigned char* b, uint32_t shard) {
        RtQueue q{};
        q.work_counter = reinterpret_cast<unsigned int*>(b);
        q.accum        = reinterpret_cast<RtFloat4*>(b + BL.off_accum);
        q.tile_first   = shard;
        q.n_tiles      = shard_tile_count(H, opt.tile_rows, shard, opt.shard_count);
        return q;
    };
    if (have_blocks) {
        P.accum        = reinterpret_cast<RtFloat4*>(own_block + BL.off_accum);
        P.work_counter = reinterpret_cast<unsigned int*>(own_block);
        uint32_t n = 0;
        P.queues[n++] = queue_of(own_block, opt.shard_index);
        if (stealing)
            for (uint32_t i = 0; i < opt.n_peer_queues; ++i) {
                const PeerQueue& pq = opt.peer_queues[i];
                if (pq.shard_index == opt.shard_index) continue;
                if (pq.shard_index >= opt.shard_count || !pq.block) throw std::runtime_error("bad peer queue entry");
                P.queues[n++] = queue_of(static_cast<unsigned char*>(pq.block), pq.shard_index);
            }
        P.n_queues = n;
    }

    // Progressive passes fused into this launch (rt_types.h): needs a fresh frame (the alpha sum tags the
    // pass) and whole-pixel items; otherwise the total is traced as one pass — the same bits either way.
    const bool fused = opt.passes > 1 && trace && !L.sample_items && !opt.accum_in &&
                       (uint64_t)opt.sample_begin + (uint64_t)opt.samples_per_pixel < (1u << 24);
    if (fused) {
        P.passes = (uint32_t)opt.passes;
        P.spp    = opt.samples_per_pixel / opt.passes;
        if (opt.resolve_each_pass) P.flags |= RT_FLAG_RESOLVE_EACH_PASS;
        if (!P.accum) {
            const size_t need = L.out_pixels * sizeof(RtFloat4);
            if (ctx.d_accum_cap < need) {
                RT_CUDA(cudaStreamSynchronize(stream));
                if (ctx.d_accum) RT_CUDA(cudaFree(ctx.d_accum));
                ctx.d_accum = nullptr; ctx.d_accum_cap = 0;
                RT_CUDA(cudaMalloc(&ctx.d_accum, need));
                ctx.d_accum_cap = need;
            }
            P.accum = ctx.d_accum;
        }
        if (have_blocks) P.queues[0].accum = P.accum;
        L.passes_fused = P.passes;
    }
    if (!have_blocks) {                                // the launch's only queue: its own shard
        P.n_queues  = 1;
        RtQueue q{};
        q.work_counter = P.work_counter; q.accum = P.accum; q.tile_first = opt.shard_index; q.n_tiles = L.n_tiles;
        P.queues[0] = q;
    }
    if ((uint64_t)slots * P.passes >= 0x7fffff00ull) throw std::runtime_error("frame shard exceeds 2^31 work slots; use more shards or fewer passes");

    // launch geometry: persistent CTAs, resident-CTA count from the occupancy API
    L.smem_limit = ctx.smem_optin > 1024 ? ctx.smem_optin - 1024 : 0;   // static smem: the mbarrier
    auto& occ    = ctx.occupancy[{scene.view.n_sph_pad, scene.view.n_tri_pad, scene.view.n_groups, opt.fast_math ? 1 : 0,
                                  opt.group_cull ? 1 : 0}];
    if (occ.per_sm == 0) {
        RT_CUDA(opt.fast_math ? occupancy_fast(scene.view, L.smem_limit, opt.group_cull, &occ.per_sm, &occ.block,
                                               &occ.hot_bytes, &occ.resident, &occ.sph_mode)
                              : occupancy_exact(scene.view, L.smem_limit, opt.group_cull, &occ.per_sm, &occ.block,
                                                &occ.hot_bytes, &occ.resident, &occ.sph_mode));
        if (occ.per_sm < 1) throw std::runtime_error("render kernel does not fit on this device");
    }
    L.hot_bytes = occ.hot_bytes;
    L.resident  = occ.resident != 0;
    L.filtered  = (occ.sph_mode & 0xff) != RT_SPH_DIRECT;
    L.culled    = (occ.sph_mode & 0xff) == RT_SPH_CULL;
    L.paths_per_lane = (uint32_t)(occ.sph_mode >> 8);
    L.block = occ.block;
    // with stealing every GPU may end up tracing any part of the frame: size the grid for the whole frame
    uint64_t frame_slots = slots;
    if (stealing) {
        frame_slots = 0;
        for (uint32_t i = 0; i < P.n_queues; ++i)
            frame_slots += (uint64_t)P.queues[i].n_tiles * ((W + 7u) / 8u) * (opt.tile_rows / 4u) * 32u;
    }
    const uint64_t work_slots = L.sample_items ? slots * (uint64_t)chunk_spp : slots * P.passes;
    const uint64_t want_ctas = ((stealing ? frame_slots * P.passes : work_slots) + (uint64_t)L.block - 1) / (uint64_t)L.block;
    L.grid = (int)std::min<uint64_t>((uint64_t)occ.per_sm * ctx.num_sms, std::max<uint64_t>(want_ctas, 1));
    // Work-queue granularity: a warp takes `reserve` pixel slots per atomicAdd.  Aim for >= 64
    // slabs per warp so that the last slab of the slowest warp is a small part of the frame.
    const uint64_t warps   = (uint64_t)L.grid * (uint64_t)(L.block / 32);
    uint64_t       reserve = work_slots / (warps * 64u) / 32u * 32u;
    P.reserve = (uint32_t)std::min<uint64_t>(std::max<uint64_t>(reserve, 32u), 256u);

    // per-tile completion flags for a host that hands tiles on while the kernel still runs (pixel items, whole frame)
    if (want_tile_flags && !L.sample_items && trace && !L.compact && opt.shard_count <= 1 && !opt.no_resolve) {
        const size_t tiles = (H + opt.tile_rows - 1) / opt.tile_rows;
        if (ctx.tile_cap < tiles) {
            RT_CUDA(cudaStreamSynchronize(stream));
            if (ctx.d_tile_done) RT_CUDA(cudaFree(ctx.d_tile_done));
            if (ctx.h_tile_flags) RT_CUDA(cudaFreeHost(ctx.h_tile_flags));
            ctx.d_tile_done = nullptr; ctx.h_tile_flags = nullptr; ctx.tile_cap = 0;
            RT_CUDA(cudaMalloc(&ctx.d_tile_done, tiles * sizeof(unsigned int)));
            RT_CUDA(cudaMallocHost(&ctx.h_tile_flags, tiles * sizeof(unsigned int)));
            std::memset(ctx.h_tile_flags, 0, tiles * sizeof(unsigned int));
            ctx.tile_cap = tiles;
            ctx.tile_epoch = 0;
        }
        if (++ctx.tile_epoch == 0u) { std::memset(ctx.h_tile_flags, 0, ctx.tile_cap * sizeof(unsigned int)); ctx.tile_epoch = 1u; }
        void* flags_dev = nullptr;
        RT_CUDA(cudaHostGetDevicePointer(&flags_dev, ctx.h_tile_flags, 0));
        RT_CUDA(cudaMemsetAsync(ctx.d_tile_done, 0, tiles * sizeof(unsigned int), stream));
        P.tile_done  = ctx.d_tile_done;
        P.tile_flags = static_cast<unsigned int*>(flags_dev);
        P.tile_epoch = ctx.tile_epoch;
        L.tile_flags = true;
    }

    // Row gather: the frame lives in another GPU's memory.  Render into a local, zeroed full frame with the very same
    // kernel, then one small kernel moves every pixel found there across NVLink as 16-byte vectors (rt_gather_rows_kernel).
    uint32_t* gather_remote = nullptr;
    if (opt.row_gather && opt.full_frame_out && opt.shard_count > 1 && !L.sample_items && trace && !opt.no_resolve &&
        !opt.resolve_each_pass && L.d_out && (L.n_tiles > 0 || stealing)) {
        const size_t px = (size_t)W * H;
        if (ctx.d_local_cap < px) {
            RT_CUDA(cudaStreamSynchronize(stream));
            if (ctx.d_local_frame) RT_CUDA(cudaFree(ctx.d_local_frame));
            ctx.d_local_frame = nullptr; ctx.d_local_cap = 0;
            RT_CUDA(cudaMalloc(&ctx.d_local_frame, px * sizeof(uint32_t)));
            ctx.d_local_cap = px;
        }
        RT_CUDA(cudaMemsetAsync(ctx.d_local_frame, 0, px * sizeof(uint32_t), stream));   // 0 = "not rendered here"
        gather_remote = L.d_out;
        P.out         = ctx.d_local_frame;
    }
    L.uses_scratch = L.sample_items || gather_remote != nullptr || (P.accum && P.accum == ctx.d_accum) || (L.d_out && L.d_out == ctx.d_out);
    if (L.n_tiles > 0 || stealing) {
        RT_CUDA(cudaMemsetAsync(L.slot, 0, sizeof(CounterSlot), stream));
        // fused passes: no stale sums may look like a finished pass.  Stream order puts this BEFORE the reset
        // of the work counter, so no other GPU can be handed a slot of this shard while its sums are cleared.
        if (fused) RT_CUDA(cudaMemsetAsync(P.accum, 0, L.out_pixels * sizeof(RtFloat4), stream));
        if (have_blocks) RT_CUDA(cudaMemsetAsync(P.work_counter, 0, sizeof(unsigned int), stream));
        if (timed) RT_CUDA(cudaEventRecord(ctx.ev0, stream));
        if (!L.sample_items) {
            RT_CUDA(opt.fast_math ? launch_render_fast(P, scene.view, L.grid, L.smem_limit, stream)
                                  : launch_render_exact(P, scene.view, L.grid, L.smem_limit, stream));
            L.launches = 1;
            if (gather_remote) {
                RT_CUDA(launch_gather_rows(ctx.d_local_frame, gather_remote, (size_t)W * H, ctx.num_sms * 4, stream));
                L.launches = 2;
            }
        } else {
            // sample items: [trace chunk_spp samples -> ordered sum] per chunk, sums handed on in P.accum
            const uint32_t user_flags = P.flags;
            const int32_t  total = opt.samples_per_pixel;
            for (int32_t done = 0; done < total; done += chunk_spp) {
                const bool first = done == 0, last = done + chunk_spp >= total;
                P.spp          = std::min(chunk_spp, total - done);
                P.sample_begin = opt.sample_begin + done;
                P.flags        = user_flags & ~(RT_FLAG_ACCUM_IN | RT_FLAG_ACCUM_OUT | RT_FLAG_NO_RESOLVE);
                if (!first || (user_flags & RT_FLAG_ACCUM_IN)) P.flags |= RT_FLAG_ACCUM_IN;
                if (!last || (user_flags & RT_FLAG_ACCUM_OUT)) P.flags |= RT_FLAG_ACCUM_OUT;
                if (!last || (user_flags & RT_FLAG_NO_RESOLVE)) P.flags |= RT_FLAG_NO_RESOLVE;
                if (!first) RT_CUDA(cudaMemsetAsync(&L.slot->work, 0, sizeof(unsigned int), stream));
                RT_CUDA(opt.fast_math ? launch_render_fast(P, scene.view, L.grid, L.smem_limit, stream)
                                      : launch_render_exact(P, scene.view, L.grid, L.smem_limit, stream));
                RT_CUDA(opt.fast_math ? launch_resolve_samples_fast(P, stream) : launch_resolve_samples_exact(P, stream));
                L.launches += 2;
            }
        }
        if (timed) RT_CUDA(cudaEventRecord(ctx.ev1, stream));
    }
    return L;
}

uint64_t shard_pixels(uint32_t W, uint32_t H, const Options& opt, uint32_t n_tiles)
{
    uint64_t px = 0;
    for (uint32_t j = 0; j < n_tiles; ++j) {
        const uint64_t tile = rt_shard_tile(opt.shard_index, opt.shard_count, j);
        const uint64_t r0   = tile * opt.tile_rows;
        const uint64_t r1   = std::min<uint64_t>(r0 + opt.tile_rows, H);
        px += (r1 - r0) * W;
    }
    return px;
}

// Staging frame -> the caller's pageable frame.  One core moves ~12 GB/s out of the freshly DMA-written (cache-cold)
// staging buffer, so large frames are split over a few threads (measured on C2, 8.3 MB: 0.70 -> see profiles/r02_bench.md).
void copy_frame(void* dst, const void* src, size_t bytes)
{
    static const unsigned workers = [] {
        const char* e = std::getenv("RT_COPY_THREADS");
        unsigned n = e ? (unsigned)std::atoi(e) : 4u;
        const unsigned hw = std::thread::hardware_concurrency();
        if (hw && n > hw) n = hw;
        return n < 1u ? 1u : n;
    }();
    if (workers == 1 || bytes < ((size_t)2 << 20)) { std::memcpy(dst, src, bytes); return; }
    const size_t piece = ((bytes + workers - 1) / workers + 4095) & ~(size_t)4095;
    std::vector<std::thread> pool;
    for (unsigned i = 1; i < workers; ++i) {
        const size_t off = (size_t)i * piece;
        if (off >= bytes) break;
        pool.emplace_back([=] { std::memcpy((char*)dst + off, (const char*)src + off, std::min(piece, bytes - off)); });
    }
    std::memcpy(dst, src, std::min(piece, bytes));
    for (auto& t : pool) t.join();
}

void ensure_stage(DeviceContext& ctx, size_t bytes)
{
    if (ctx.h_stage_cap >= bytes) return;
    if (ctx.h_stage) RT_CUDA(cudaFreeHost(ctx.h_stage));
    ctx.h_stage = nullptr; ctx.h_stage_cap = 0;
    RT_CUDA(cudaMallocHost(&ctx.h_stage, bytes));
    ctx.h_stage_cap = bytes;
}

}   // namespace

void ray_trace_into(const World& world, const Camera& camera, size_t width, size_t height,
                    const Options& opt, ColorU8* host_pixels, void* device_pixels, void* device_accum,
                    void* user_stream)
{
    const auto t_begin = std::chrono::steady_clock::now();
    std::lock_guard<std::mutex> lock(g_mutex);
    validate(width, height, opt, device_accum);

    const int   dev = resolve_device(opt.device);
    DeviceGuard guard(dev);                  // the caller's current device is restored on every exit path
    DeviceContext&     ctx   = context_for(dev);
    const DeviceScene& scene = device_scene(world, ctx);
    cudaStream_t       stream = user_stream ? static_cast<cudaStream_t>(user_stream) : ctx.stream;

    const uint32_t W = (uint32_t)width, H = (uint32_t)height;
    // Pinned destination (rt_alloc_pixels, cudaHostRegister): the kernel stores every finished
    // pixel straight into the caller's frame over PCIe (mapped host memory) — 4 B per pixel spread
    // over the whole render, so no D2H copy follows the kernel.
    // Only when the kernel runs long enough to hide them: 32-byte PCIe writes sustain ~7 GB/s (measured:
    // a 1-spp 1080p frame takes 1.27 ms this way against 0.37 ms with the copy), a D2H copy ~50 GB/s.
    const uint64_t work_per_pixel = (uint64_t)std::max(opt.samples_per_pixel, 0) *
                                    ((uint64_t)scene.view.n_sph + scene.view.n_tri + 8u);
    const bool want_zero_copy = host_pixels && !device_pixels && !opt.no_resolve && work_per_pixel >= 256u;
    void*      zero_copy      = want_zero_copy ? mapped_device_pointer(host_pixels) : nullptr;
    // Pageable destination (what the reference's callers pass: UnsafeMutablePointer.allocate in
    // GameView.swift:125-129, a Vec in examples/c_raytracer.rs:53): the kernel stores its pixels into the
    // library's pinned staging frame the same way, and one memcpy hands them over — no D2H copy either.
    // RT_PAGEABLE selects the way to a pageable frame (A/B measurements): zc = staged zero-copy (default),
    // d2h = one D2H into the staging frame then memcpy, chunk = D2H in pieces overlapped with their memcpy.
    static const int pageable_mode = [] {
        const char* e = std::getenv("RT_PAGEABLE");
        if (!e) return 0;
        return !std::strcmp(e, "d2h") ? 1 : !std::strcmp(e, "chunk") ? 2 : 0;
    }();
    bool staged_zero_copy = false;
    if (pageable_mode == 0 && want_zero_copy && !zero_copy && !is_pinned_or_device_accessible(host_pixels)) {
        ensure_stage(ctx, (size_t)W * H * 4);
        zero_copy = mapped_device_pointer(ctx.h_stage);
        staged_zero_copy = zero_copy != nullptr;
    }
    Options       zc_opt = opt;
    if (zero_copy) zc_opt.full_frame_out = true;            // tiles land at their frame offsets
    const ShardLaunch L = enqueue_shard(ctx, scene, camera, W, H, zero_copy ? zc_opt : opt,
                                        zero_copy ? static_cast<uint32_t*>(zero_copy) : static_cast<uint32_t*>(device_pixels),
                                        device_accum, stream, opt.stats != nullptr, staged_zero_copy);
    const uint32_t n_tiles = L.n_tiles;
    uint32_t*      d_out   = L.d_out;

    if (zero_copy && L.tile_flags) {
        // The kernel flags every finished 16-row tile (bottom rows first); its rows go from the staging frame to the
        // caller's frame while the rest is still being rendered, so that only the last tile's copy follows the kernel.
        const size_t tiles = (H + opt.tile_rows - 1) / opt.tile_rows, tile_bytes = (size_t)opt.tile_rows * W * 4;
        const volatile unsigned int* flags = ctx.h_tile_flags;
        std::vector<unsigned char> copied(tiles, 0);
        size_t left = tiles;
        bool   finished = false;
        while (left) {
            size_t progressed = 0;
            for (size_t t = tiles; t-- > 0;) {
                if (copied[t] || flags[t] != ctx.tile_epoch) continue;
                std::atomic_thread_fence(std::memory_order_acquire);
                const size_t off = t * tile_bytes, cnt = std::min(tile_bytes, (size_t)W * H * 4 - off);
                std::memcpy(reinterpret_cast<unsigned char*>(host_pixels) + off, ctx.h_stage + off, cnt);
                copied[t] = 1; --left; ++progressed;
            }
            if (left && !progressed) {
                if (finished) throw std::runtime_error("render kernel finished without completing every tile");
                const cudaError_t q = cudaStreamQuery(stream);
                if (q == cudaSuccess) finished = true;             // one more sweep picks up the last flags
                else if (q != cudaErrorNotReady) fail("render kernel", q);
            }
        }
        RT_CUDA(cudaStreamSynchronize(stream));
    } else if (zero_copy) {
        RT_CUDA(cudaStreamSynchronize(stream));
        if (staged_zero_copy) {              // this shard's rows of the staging frame -> the caller's frame
            const size_t tile_px = (size_t)opt.tile_rows * W;
            if (opt.shard_count <= 1) {
                copy_frame(host_pixels, ctx.h_stage, (size_t)W * H * 4);
            } else {
                for (uint32_t j = 0; j < n_tiles; ++j) {
                    const size_t first = (size_t)rt_shard_tile(opt.shard_index, opt.shard_count, j) * tile_px;
                    const size_t count = std::min(tile_px, (size_t)W * H - first);
                    std::memcpy(reinterpret_cast<unsigned char*>(host_pixels) + first * 4, ctx.h_stage + first * 4, count * 4);
                }
            }
        }
    } else if (host_pixels && !opt.no_resolve && n_tiles > 0) {
        // D2H of the finished RGBA8 rows.  Every tile is one contiguous byte range of the frame
        // (image.rs:27 row-major), so a shard copies tile by tile and a full frame in one piece.
        const bool   direct  = is_pinned_or_device_accessible(host_pixels);
        const size_t tile_px = (size_t)opt.tile_rows * W;
        uint32_t*    host32  = reinterpret_cast<uint32_t*>(host_pixels);
        if (!direct) ensure_stage(ctx, L.out_pixels * 4);
        // (frame offset, device offset, count) of every contiguous piece this shard owns
        auto for_each_piece = [&](auto&& f) {
            if (opt.shard_count <= 1) { f((size_t)0, (size_t)0, (size_t)W * H); return; }
            for (uint32_t j = 0; j < n_tiles; ++j) {
                const size_t tile  = rt_shard_tile(opt.shard_index, opt.shard_count, j);
                const size_t first = tile * tile_px;
                const size_t count = std::min(tile_px, (size_t)W * H - first);
                f(first, L.compact ? (size_t)j * tile_px : first, count);
            }
        };
        if (!direct && pageable_mode == 2 && opt.shard_count <= 1) {
            // pieces of ~1 MiB: the memcpy of piece i runs while pieces i+1.. are still on their way
            const size_t total = (size_t)W * H * 4, piece = (size_t)1 << 20;
            const size_t n = (total + piece - 1) / piece;
            while (ctx.ev_chunk.size() < n) {
                cudaEvent_t e;
                RT_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
                ctx.ev_chunk.push_back(e);
            }
            const unsigned char* src = reinterpret_cast<const unsigned char*>(d_out);
            for (size_t i = 0; i < n; ++i) {
                const size_t off = i * piece, cnt = std::min(piece, total - off);
                RT_CUDA(cudaMemcpyAsync(ctx.h_stage + off, src + off, cnt, cudaMemcpyDeviceToHost, stream));
                RT_CUDA(cudaEventRecord(ctx.ev_chunk[i], stream));
            }
            for (size_t i = 0; i < n; ++i) {
                const size_t off = i * piece, cnt = std::min(piece, total - off);
                RT_CUDA(cudaEventSynchronize(ctx.ev_chunk[i]));
                std::memcpy(reinterpret_cast<unsigned char*>(host_pixels) + off, ctx.h_stage + off, cnt);
            }
        } else {
        for_each_piece([&](size_t frame_px, size_t dev_px, size_t count) {
            void* dst = direct ? (void*)(host32 + frame_px) : (void*)(ctx.h_stage + dev_px * 4);
            RT_CUDA(cudaMemcpyAsync(dst, d_out + dev_px, count * 4, cudaMemcpyDeviceToHost, stream));
        });
        RT_CUDA(cudaStreamSynchronize(stream));
        if (!direct)
            for_each_piece([&](size_t frame_px, size_t dev_px, size_t count) {
                copy_frame(host32 + frame_px, ctx.h_stage + dev_px * 4, count * 4);
            });
        }
    } else if (!user_stream || L.uses_scratch) {
        // A caller's stream normally gets the work enqueued and the call returns; but the per-device scratch (sample
        // buffer of the sample-item mode, hand-over sums, internal frame) is shared by every launch on the device, so
        // a launch that uses it is finished before the next one — possibly on another stream — may be enqueued.
        RT_CUDA(cudaStreamSynchronize(stream));
    }

    if (opt.stats) {
        RenderStats& st = *opt.stats;
        st = RenderStats{};
        st.grid       = (uint32_t)L.grid;
        st.block      = (uint32_t)L.block;
        st.resident   = L.resident ? 1u : 0u;
        st.smem_bytes = st.resident ? (uint32_t)L.hot_bytes : 0u;
        st.filtered   = L.filtered ? 1u : 0u;
        st.culled     = L.culled ? 1u : 0u;
        if (n_tiles > 0) {
            RT_CUDA(cudaMemcpyAsync(ctx.h_slot, L.slot, sizeof(CounterSlot), cudaMemcpyDeviceToHost, stream));
            RT_CUDA(cudaStreamSynchronize(stream));
            RT_CUDA(cudaEventElapsedTime(&st.kernel_ms, ctx.ev0, ctx.ev1));
            st.rays     = ctx.h_slot->rays;
            st.stolen_slots = ctx.h_slot->stolen;
            st.passes_fused = L.passes_fused;
            st.paths_per_lane = L.paths_per_lane;
            st.launches = L.launches;
            st.sample_items = L.sample_items ? 1u : 0u;
            st.samples  = (opt.samples_per_pixel > 0 && opt.max_ray_bounces > 0)
                              ? shard_pixels(W, H, opt, n_tiles) * (uint64_t)opt.samples_per_pixel : 0;
        }
        st.total_ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t_begin).count();
    }
}

void render_aov(const World& world, const Camera& camera, size_t width, size_t height, const Options& opt,
                const AovBuffers& buf, void* user_stream)
{
    const auto t_begin = std::chrono::steady_clock::now();
    // host-side checks, before any device work: the options this call cannot honour ...
    auto reject = [](const char* what) { throw std::runtime_error(std::string("render_aov: ") + what); };
    if (opt.fast_math) reject("RT_OPT_FAST_MATH is not supported (the buffers are exact World::hit records)");
    if (opt.accum_in || opt.accum_out) reject("RT_OPT_ACCUM_IN / RT_OPT_ACCUM_OUT are not supported (no colour sums)");
    if (opt.no_resolve || opt.resolve_each_pass) reject("RT_OPT_NO_RESOLVE / RT_OPT_RESOLVE_EACH_PASS are not supported (no RGBA8 frame)");
    if (opt.full_frame_out || opt.row_gather || opt.no_steal)
        reject("RT_OPT_FULL_FRAME_OUT / RT_OPT_ROW_GATHER / RT_OPT_NO_STEAL are not supported (single device, whole frame)");
    if (opt.shard_count > 1) reject("shard_count > 1 is not supported (single device, whole frame)");
    if (opt.n_devices > 1) reject("n_devices > 1 is not supported (single device, whole frame)");
    if (opt.passes > 1) reject("passes > 1 is not supported (one ray per pixel)");
    if (opt.peer_queues || opt.n_peer_queues) reject("peer_queues are not supported (single device, whole frame)");
    // ... the buffers and the frame size
    const float* ptrs[5] = {buf.depth, buf.position, buf.normal, buf.albedo, reinterpret_cast<const float*>(buf.prim)};
    static const char* const names[5] = {"depth", "position", "normal", "albedo", "prim"};
    if (!ptrs[0] && !ptrs[1] && !ptrs[2] && !ptrs[3] && !ptrs[4]) reject("every buffer is NULL");
    validate_size(width, height);
    if (((width + 7u) / 8u) * ((height + 3u) / 4u) >= 0x80000000ull) reject("frame exceeds 2^31 sub-tiles of 8x4 pixels");

    std::lock_guard<std::mutex> lock(g_mutex);
    const int   dev = resolve_device(opt.device);
    DeviceGuard guard(dev);                  // the caller's current device is restored on every exit path
    for (int k = 0; k < 5; ++k) {
        if (!ptrs[k]) continue;
        cudaPointerAttributes a;
        const cudaError_t     e = cudaPointerGetAttributes(&a, ptrs[k]);
        if (e != cudaSuccess) cudaGetLastError();
        if (e != cudaSuccess || a.type != cudaMemoryTypeDevice || a.device != dev)
            throw std::runtime_error(std::string("render_aov: the ") + names[k] + " buffer is not device memory of device " +
                                     std::to_string(dev));
    }
    DeviceContext&     ctx    = context_for(dev);
    const DeviceScene& scene  = device_scene(world, ctx);
    cudaStream_t       stream = user_stream ? static_cast<cudaStream_t>(user_stream) : ctx.stream;

    const uint32_t W = (uint32_t)width, H = (uint32_t)height;
    RtAovParams A{};
    A.camera       = camera.d;
    A.wm1          = (float)(W - 1u);        // `(width - 1) as f32`, common.rs:335
    A.hm1          = (float)(H - 1u);
    A.width        = W;
    A.height       = H;
    A.seed         = opt.seed;
    A.sample_begin = opt.sample_begin;
    A.flags        = opt.fixed_jitter ? RT_FLAG_FIXED_JITTER : 0u;
    A.one          = 1.0f;
    A.depth = buf.depth; A.position = buf.position; A.normal = buf.normal; A.albedo = buf.albedo; A.prim = buf.prim;

    // launch geometry: persistent CTAs, resident-CTA count from the occupancy API (cached per scene shape)
    const size_t smem_limit = ctx.smem_optin > 1024 ? ctx.smem_optin - 1024 : 0;   // static smem: the mbarrier
    auto& occ = ctx.aov_occupancy[{scene.view.n_sph_pad, scene.view.n_tri_pad, scene.view.n_groups, opt.group_cull ? 1 : 0}];
    if (occ.per_sm == 0) {
        RT_CUDA(aov_occupancy_exact(scene.view, smem_limit, opt.group_cull, &occ.per_sm, &occ.block, &occ.hot_bytes,
                                    &occ.resident, &occ.sph_mode));
        if (occ.per_sm < 1) throw std::runtime_error("first-hit kernel does not fit on this device");
    }
    const uint64_t threads = ((uint64_t)(W + 7u) / 8u) * ((H + 3u) / 4u) * 32u;
    const int      grid    = (int)std::min<uint64_t>((uint64_t)occ.per_sm * ctx.num_sms,
                                                     std::max<uint64_t>((threads + occ.block - 1) / occ.block, 1));
    if (opt.stats) RT_CUDA(cudaEventRecord(ctx.ev0, stream));
    RT_CUDA(launch_aov_exact(A, scene.view, opt.group_cull, grid, smem_limit, stream));
    if (opt.stats) RT_CUDA(cudaEventRecord(ctx.ev1, stream));
    if (!user_stream || opt.stats) RT_CUDA(cudaStreamSynchronize(stream));

    if (opt.stats) {
        RenderStats& st = *opt.stats;
        st = RenderStats{};
        RT_CUDA(cudaEventElapsedTime(&st.kernel_ms, ctx.ev0, ctx.ev1));
        st.rays       = (uint64_t)W * H;          // one World::hit per pixel
        st.samples    = (uint64_t)W * H;
        st.launches   = 1;
        st.grid       = (uint32_t)grid;
        st.block      = (uint32_t)occ.block;
        st.resident   = occ.resident ? 1u : 0u;
        st.smem_bytes = st.resident ? (uint32_t)occ.hot_bytes : 0u;
        st.filtered   = occ.sph_mode != RT_SPH_DIRECT ? 1u : 0u;
        st.culled     = occ.sph_mode == RT_SPH_CULL ? 1u : 0u;
        st.total_ms   = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t_begin).count();
    }
}

namespace {

// The host side the two ray calls share (trace_rays, occluded_rays).  `call` prefixes every rejection; out[] are the
// call's outputs with their byte counts for n rays; `all_null` is the rejection when every output is NULL.  Checks the
// arguments before any device work, then the memory, looks up the context and the scene, sizes the persistent grid
// from the kernel's cached occupancy, runs launch(scene, smem_limit, grid, stream) and fills the stats.
struct RayOutput { const void* ptr; uint64_t bytes; const char* name; };
using OccupancyMap = std::map<std::tuple<uint32_t, uint32_t, uint32_t, int>, DeviceContext::Geometry> DeviceContext::*;
using OccupancyFn  = cudaError_t (*)(const RtSceneView&, size_t, bool, int*, int*, size_t*, int*, int*);

template <class Launch>
void ray_query(const char* call, const RayQueryOptions& opt, const World& world, size_t n, const void* rays,
               const RayOutput* out, int n_out, const char* all_null, OccupancyMap cache, OccupancyFn occupancy,
               const char* kernel_name, void* user_stream, Launch&& launch)
{
    const auto t_begin = std::chrono::steady_clock::now();
    // host-side checks, before any device work
    const std::string prefix = std::string(call) + ": ";
    auto reject = [&](const std::string& what) { throw std::runtime_error(prefix + what); };
    if (n == 0) reject("n must be at least 1");
    if (n > 0x7fffffffu) reject("n must be at most 2^31 - 1");
    if (!rays) reject("the ray buffer is NULL");
    if (reinterpret_cast<uintptr_t>(rays) & 15u) reject("the ray buffer is not 16-byte aligned");
    bool any = false;
    for (int k = 0; k < n_out; ++k) any = any || out[k].ptr;
    if (!any) reject(all_null);
    auto overlaps = [](const void* a, uint64_t na, const void* b, uint64_t nb) {
        const uintptr_t x = reinterpret_cast<uintptr_t>(a), y = reinterpret_cast<uintptr_t>(b);
        return x < y + nb && y < x + na;
    };
    for (int k = 0; k < n_out; ++k) {
        if (!out[k].ptr) continue;
        if (overlaps(out[k].ptr, out[k].bytes, rays, 32ull * n)) reject(std::string("the ") + out[k].name + " output overlaps the rays");
        for (int j = 0; j < k; ++j)
            if (out[j].ptr && overlaps(out[k].ptr, out[k].bytes, out[j].ptr, out[j].bytes))
                reject(std::string("the ") + out[k].name + " output overlaps the " + out[j].name + " output");
    }

    std::lock_guard<std::mutex> lock(g_mutex);
    const int   dev = resolve_device(opt.device);
    DeviceGuard guard(dev);                  // the caller's current device is restored on every exit path
    for (int k = -1; k < n_out; ++k) {
        const void* p = k < 0 ? rays : out[k].ptr;
        if (!p) continue;
        cudaPointerAttributes a;
        const cudaError_t     e = cudaPointerGetAttributes(&a, p);
        if (e != cudaSuccess) cudaGetLastError();
        if (e != cudaSuccess || a.type != cudaMemoryTypeDevice || a.device != dev)
            reject(std::string("the ") + (k < 0 ? "ray" : out[k].name) + " buffer is not device memory of device " +
                   std::to_string(dev));
    }
    DeviceContext&     ctx    = context_for(dev);
    const DeviceScene& scene  = device_scene(world, ctx);
    cudaStream_t       stream = user_stream ? static_cast<cudaStream_t>(user_stream) : ctx.stream;

    // launch geometry: persistent CTAs, resident-CTA count from the occupancy API (cached per kernel and scene shape)
    const size_t smem_limit = ctx.smem_optin > 1024 ? ctx.smem_optin - 1024 : 0;   // static smem: the mbarrier
    auto& occ = (ctx.*cache)[{scene.view.n_sph_pad, scene.view.n_tri_pad, scene.view.n_groups, opt.group_cull ? 1 : 0}];
    if (occ.per_sm == 0) {
        RT_CUDA(occupancy(scene.view, smem_limit, opt.group_cull, &occ.per_sm, &occ.block, &occ.hot_bytes, &occ.resident,
                          &occ.sph_mode));
        if (occ.per_sm < 1) throw std::runtime_error(std::string(kernel_name) + " does not fit on this device");
    }
    const uint64_t threads = ((uint64_t)n + 31u) / 32u * 32u;
    const int      grid    = (int)std::min<uint64_t>((uint64_t)occ.per_sm * ctx.num_sms,
                                                     std::max<uint64_t>((threads + occ.block - 1) / occ.block, 1));
    if (opt.stats) RT_CUDA(cudaEventRecord(ctx.ev0, stream));
    RT_CUDA(launch(scene.view, smem_limit, grid, stream));
    if (opt.stats) RT_CUDA(cudaEventRecord(ctx.ev1, stream));
    if (!user_stream || opt.stats) RT_CUDA(cudaStreamSynchronize(stream));

    if (opt.stats) {
        RenderStats& st = *opt.stats;
        st = RenderStats{};
        RT_CUDA(cudaEventElapsedTime(&st.kernel_ms, ctx.ev0, ctx.ev1));
        st.rays       = n;                        // one walk per ray
        st.samples    = n;
        st.launches   = 1;
        st.grid       = (uint32_t)grid;
        st.block      = (uint32_t)occ.block;
        st.resident   = occ.resident ? 1u : 0u;
        st.smem_bytes = st.resident ? (uint32_t)occ.hot_bytes : 0u;
        st.filtered   = occ.sph_mode != RT_SPH_DIRECT ? 1u : 0u;
        st.culled     = occ.sph_mode == RT_SPH_CULL ? 1u : 0u;
        st.total_ms   = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t_begin).count();
    }
}

}   // namespace

void trace_rays(const World& world, const RayQueryOptions& opt, size_t n, const void* rays, const AovBuffers& buf,
                void* user_stream)
{
    const RayOutput out[5] = {{buf.depth, 4ull * n, "depth"}, {buf.position, 12ull * n, "position"},
                              {buf.normal, 12ull * n, "normal"}, {buf.albedo, 12ull * n, "albedo"},
                              {buf.prim, 4ull * n, "prim"}};
    ray_query("trace_rays", opt, world, n, rays, out, 5, "every output is NULL", &DeviceContext::ray_occupancy,
              rays_occupancy_exact, "ray-query kernel", user_stream,
              [&](const RtSceneView& G, size_t smem_limit, int grid, cudaStream_t stream) {
                  RtRayParams R{};
                  R.rays = static_cast<const RtFloat4*>(rays);
                  R.n    = (uint32_t)n;
                  R.one  = 1.0f;
                  R.depth = buf.depth; R.position = buf.position; R.normal = buf.normal; R.albedo = buf.albedo; R.prim = buf.prim;
                  return launch_rays_exact(R, G, opt.group_cull, grid, smem_limit, stream);
              });
}

void occluded_rays(const World& world, const RayQueryOptions& opt, size_t n, const void* rays, uint8_t* occluded,
                   void* user_stream)
{
    const RayOutput out[1] = {{occluded, n, "occluded"}};
    ray_query("occluded_rays", opt, world, n, rays, out, 1, "the occluded output is NULL",
              &DeviceContext::occlusion_occupancy, occlusion_occupancy_exact, "occlusion kernel", user_stream,
              [&](const RtSceneView& G, size_t smem_limit, int grid, cudaStream_t stream) {
                  RtOcclusionParams Q{};
                  Q.rays     = static_cast<const RtFloat4*>(rays);
                  Q.n        = (uint32_t)n;
                  Q.one      = 1.0f;
                  Q.occluded = occluded;
                  return launch_occlusion_exact(Q, G, opt.group_cull, grid, smem_limit, stream);
              });
}

void denoise(const DenoiseOptions& opt, size_t width, size_t height, int32_t spp, const DenoiseBuffers& buf,
             void* user_stream)
{
    const auto t_begin = std::chrono::steady_clock::now();
    // host-side checks, before any device work
    auto reject = [](const std::string& what) { throw std::runtime_error("denoise: " + what); };
    if (opt.iterations > kDenoiseMaxIterations) reject("iterations must be in 1..10 (0: the default, 5)");
    const float sigmas[3] = {opt.sigma_color, opt.sigma_normal, opt.sigma_plane};
    static const char* const sigma_names[3] = {"sigma_color", "sigma_normal", "sigma_plane"};
    for (int k = 0; k < 3; ++k)
        if (!(sigmas[k] >= 0.0f) || std::isinf(sigmas[k]))
            reject(std::string(sigma_names[k]) + " must be finite and > 0 (0: the default)");
    if (spp < 1) reject("spp must be >= 1");
    const void* in[5] = {buf.accum, buf.normal, buf.position, buf.albedo, buf.prim};
    static const char* const in_names[5] = {"accum", "normal", "position", "albedo", "prim"};
    for (int k = 0; k < 5; ++k)
        if (!in[k]) reject(std::string("the ") + in_names[k] + " buffer is NULL (required)");
    if (!buf.pixels && !buf.color) reject("both outputs (pixels, color) are NULL");
    try { validate_size(width, height); } catch (const std::runtime_error& e) { reject(e.what()); }
    const uint64_t n = (uint64_t)width * height;
    const uint64_t in_bytes[5] = {16 * n, 12 * n, 12 * n, 12 * n, 4 * n};
    const void*    out[2] = {buf.pixels, buf.color};
    static const char* const out_names[2] = {"pixels", "color"};
    const uint64_t out_bytes[2] = {4 * n, 16 * n};
    auto overlaps = [](const void* a, uint64_t na, const void* b, uint64_t nb) {
        const uintptr_t x = reinterpret_cast<uintptr_t>(a), y = reinterpret_cast<uintptr_t>(b);
        return x < y + nb && y < x + na;
    };
    for (int o = 0; o < 2; ++o) {
        if (!out[o]) continue;
        for (int k = 0; k < 5; ++k)
            if (overlaps(out[o], out_bytes[o], in[k], in_bytes[k]))
                reject(std::string("the ") + out_names[o] + " output overlaps the " + in_names[k] + " input");
    }
    if (out[0] && out[1] && overlaps(out[0], out_bytes[0], out[1], out_bytes[1])) reject("the two outputs overlap");

    std::lock_guard<std::mutex> lock(g_mutex);
    const int   dev = resolve_device(opt.device);
    DeviceGuard guard(dev);                  // the caller's current device is restored on every exit path
    for (int k = 0; k < 7; ++k) {
        const void* p = k < 5 ? in[k] : out[k - 5];
        if (!p) continue;
        cudaPointerAttributes a;
        const cudaError_t     e = cudaPointerGetAttributes(&a, p);
        if (e != cudaSuccess) cudaGetLastError();
        if (e != cudaSuccess || a.type != cudaMemoryTypeDevice || a.device != dev)
            throw std::runtime_error(std::string("denoise: the ") + (k < 5 ? in_names[k] : out_names[k - 5]) +
                                     " buffer is not device memory of device " + std::to_string(dev));
    }
    DeviceContext& ctx    = context_for(dev);
    cudaStream_t   stream = user_stream ? static_cast<cudaStream_t>(user_stream) : ctx.stream;

    // scratch: two demodulated colour frames and the packed guides, 64 B per pixel, grown on demand.  Every call that
    // uses it returns only after its work is finished (below), so the scratch is idle whenever a call starts.
    const size_t need = (size_t)n * 4;
    if (ctx.d_denoise_cap < need) {
        if (ctx.d_denoise) RT_CUDA(cudaFree(ctx.d_denoise));
        ctx.d_denoise     = nullptr;
        ctx.d_denoise_cap = 0;
        RT_CUDA(cudaMalloc(&ctx.d_denoise, need * sizeof(RtFloat4)));
        ctx.d_denoise_cap = need;
    }

    RtDenoiseParams P{};
    P.accum      = static_cast<const RtFloat4*>(buf.accum);
    P.normal     = buf.normal;
    P.position   = buf.position;
    P.albedo     = buf.albedo;
    P.prim       = buf.prim;
    P.pixels     = static_cast<uint32_t*>(buf.pixels);
    P.color      = static_cast<RtFloat4*>(buf.color);
    P.e[0]       = ctx.d_denoise;
    P.e[1]       = ctx.d_denoise + n;
    P.gn         = ctx.d_denoise + 2 * n;
    P.gx         = ctx.d_denoise + 3 * n;
    P.width      = (uint32_t)width;
    P.height     = (uint32_t)height;
    P.iterations = opt.iterations ? opt.iterations : kDenoiseDefaultIterations;
    P.k          = 1.0f / (float)spp;                     // resolve_pixel's reciprocal
    auto scale = [](float sigma) { return 1.0f / ((16.0f * sigma) * sigma); };   // rt_denoise.cuh dn_scale
    P.sc         = scale(opt.sigma_color > 0.0f ? opt.sigma_color : kDenoiseDefaultSigmaColor);
    P.sn         = scale(opt.sigma_normal > 0.0f ? opt.sigma_normal : kDenoiseDefaultSigmaNormal);
    P.sx         = scale(opt.sigma_plane > 0.0f ? opt.sigma_plane : kDenoiseDefaultSigmaPlane);

    uint32_t grid = 0, block = 0;
    if (opt.stats) RT_CUDA(cudaEventRecord(ctx.ev0, stream));
    RT_CUDA(launch_denoise(P, ctx.num_sms, &grid, &block, stream));
    if (opt.stats) RT_CUDA(cudaEventRecord(ctx.ev1, stream));
    RT_CUDA(cudaStreamSynchronize(stream));      // the scratch is shared by every call on the device

    if (opt.stats) {
        RenderStats& st = *opt.stats;
        st = RenderStats{};
        RT_CUDA(cudaEventElapsedTime(&st.kernel_ms, ctx.ev0, ctx.ev1));
        st.rays     = 0;
        st.samples  = 0;
        st.launches = 1 + P.iterations;
        st.grid     = grid;
        st.block    = block;
        st.total_ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t_begin).count();
    }
}

// One process, several GPUs (the shape the C-ABI callers have: GameView.swift and
// examples/c_raytracer.rs are single processes).  Device d renders row tiles d, d+N, ... and
// its kernel stores the finished RGBA8 pixels DIRECTLY into device 0's frame through a
// peer mapping (NVLink/NVSwitch): the gather of SURVEY.md 8e is fused into the pack step, no
// separate collective or copy exists.  Device 0 then sends the frame to the host once.
// Without peer access the shards fall back to one D2H per tile from every device.
void ray_trace_multi(const World& world, const Camera& camera, size_t width, size_t height, const Options& opt_in,
                     ColorU8* host_pixels, int n_devices)
{
    const auto t_begin = std::chrono::steady_clock::now();
    if (!host_pixels) throw std::runtime_error("ray_trace_multi: host_pixels is null");
    if (opt_in.accum_in || opt_in.accum_out || opt_in.no_resolve)
        throw std::runtime_error("ray_trace_multi: progressive passes are per-device (use rt_render_device)");
    int avail = 0;
    {
        cudaError_t e = cudaGetDeviceCount(&avail);
        if (e != cudaSuccess || avail == 0)
            throw std::runtime_error("no CUDA device available (this library has no CPU render path)");
    }
    const int N = std::min(n_devices, avail);
    if (N <= 1) {
        Options o = opt_in;
        o.device = 0; o.shard_index = 0; o.shard_count = 1; o.full_frame_out = false;
        o.peer_queues = nullptr; o.n_peer_queues = 0;
        ray_trace_into(world, camera, width, height, o, host_pixels, nullptr, nullptr, nullptr);
        return;
    }
    std::unique_lock<std::mutex> lock(g_mutex);
    int caller_device = -1;
    if (cudaGetDevice(&caller_device) != cudaSuccess) { cudaGetLastError(); caller_device = -1; }
    struct Restore { int d; ~Restore() { if (d >= 0) cudaSetDevice(d); } } restore{caller_device};
    Options base = opt_in;
    base.shard_count = (uint32_t)N;
    base.peer_queues = nullptr; base.n_peer_queues = 0;
    validate(width, height, base, nullptr);
    const uint32_t W = (uint32_t)width, H = (uint32_t)height;

    // contexts, scenes, peer access: to device 0 for the fused gather, all-to-all for work stealing
    std::vector<DeviceContext*> ctxs(N);
    bool peer = true, all_peer = N <= (int)RT_MAX_QUEUES;
    for (int d = 0; d < N; ++d) {
        RT_CUDA(cudaSetDevice(d));
        ctxs[d] = &context_for(d);
        (void)device_scene(world, *ctxs[d]);
        for (int e = 0; e < N; ++e) {
            if (e == d) continue;
            int can = 0;
            RT_CUDA(cudaDeviceCanAccessPeer(&can, d, e));
            if (can) {
                cudaError_t err = cudaDeviceEnablePeerAccess(e, 0);
                if (err != cudaSuccess && err != cudaErrorPeerAccessAlreadyEnabled) fail("cudaDeviceEnablePeerAccess", err);
                cudaGetLastError();
            } else {
                all_peer = false;
                if (e == 0) peer = false;
            }
        }
    }
    static const bool steal_enabled = [] { const char* e = std::getenv("RT_STEAL"); return !(e && *e == '0'); }();
    const bool steal = peer && all_peer;               // shard blocks (work counters + sums) reachable from every device
    DeviceContext& c0 = *ctxs[0];
    RT_CUDA(cudaSetDevice(0));
    if (c0.d_out_cap < (size_t)W * H) {
        RT_CUDA(cudaStreamSynchronize(c0.stream));
        if (c0.d_out) RT_CUDA(cudaFree(c0.d_out));
        c0.d_out = nullptr; c0.d_out_cap = 0;
        RT_CUDA(cudaMalloc(&c0.d_out, (size_t)W * H * sizeof(uint32_t)));
        c0.d_out_cap = (size_t)W * H;
    }
    // shard blocks: every device's work counter (+ the sums of fused passes), reachable from all the others
    std::vector<PeerQueue> blocks;
    if (steal) {
        const size_t need = base.passes > 1 ? shard_block_bytes(W, H) : kBlockHeader;
        for (int d = 0; d < N; ++d) {
            DeviceContext& c = *ctxs[d];
            if (c.d_block_cap < need) {
                RT_CUDA(cudaSetDevice(d));
                RT_CUDA(cudaStreamSynchronize(c.stream));
                if (c.d_block) RT_CUDA(cudaFree(c.d_block));
                c.d_block = nullptr; c.d_block_cap = 0;
                RT_CUDA(cudaMalloc(&c.d_block, need));
                c.d_block_cap = need;
                shard_block_init(c.d_block);
            }
        }
        blocks.resize(N);
    }

    std::vector<ShardLaunch> launches(N);
    const bool   direct  = is_pinned_or_device_accessible(host_pixels);
    uint32_t*    host32  = reinterpret_cast<uint32_t*>(host_pixels);
    const size_t tile_px = (size_t)base.tile_rows * W;
    for (int d = 0; d < N; ++d) {
        RT_CUDA(cudaSetDevice(d));
        Options o = base;
        o.device = d; o.shard_index = (uint32_t)d; o.full_frame_out = peer;
        static const bool row_gather_enabled = [] { const char* e = std::getenv("RT_ROW_GATHER"); return !(e && *e == '0'); }();
        o.row_gather = peer && d > 0 && row_gather_enabled;    // device 0 writes its own memory
        if (steal) {                                   // raid order: the next device first, so that the thieves spread
            for (int i = 0; i < N; ++i) {
                const int e = (d + i) % N;
                blocks[i] = PeerQueue{ctxs[e]->d_block, (uint32_t)e, 0u};
            }
            o.peer_queues = blocks.data(); o.n_peer_queues = (uint32_t)N;
            o.no_steal    = !steal_enabled;
        }
        launches[d] = enqueue_shard(*ctxs[d], device_scene(world, *ctxs[d]), camera, W, H, o,
                                    peer ? c0.d_out : nullptr, nullptr, ctxs[d]->stream, true);
        if (!peer && launches[d].n_tiles > 0) {        // fallback gather: D2H tile by tile from every device
            if (!direct) ensure_stage(*ctxs[d], launches[d].out_pixels * 4);
            for (uint32_t j = 0; j < launches[d].n_tiles; ++j) {
                const size_t first = (size_t)rt_shard_tile((uint32_t)d, (uint32_t)N, j) * tile_px;
                const size_t count = std::min(tile_px, (size_t)W * H - first);
                void* dst = direct ? (void*)(host32 + first) : (void*)(ctxs[d]->h_stage + (size_t)j * tile_px * 4);
                RT_CUDA(cudaMemcpyAsync(dst, launches[d].d_out + (size_t)j * tile_px, count * 4, cudaMemcpyDeviceToHost,
                                        ctxs[d]->stream));
            }
        }
    }
    // wait for every device; with peer stores the frame is then complete in device 0's memory
    for (int d = N - 1; d >= 0; --d) {
        RT_CUDA(cudaSetDevice(d));
        RT_CUDA(cudaStreamSynchronize(ctxs[d]->stream));
        if (!peer && !direct)
            for (uint32_t j = 0; j < launches[d].n_tiles; ++j) {
                const size_t first = (size_t)rt_shard_tile((uint32_t)d, (uint32_t)N, j) * tile_px;
                const size_t count = std::min(tile_px, (size_t)W * H - first);
                std::memcpy(host32 + first, ctxs[d]->h_stage + (size_t)j * tile_px * 4, count * 4);
            }
    }
    if (peer) {                                        // device 0 is current here
        void* dst = host32;
        if (!direct) { ensure_stage(c0, (size_t)W * H * 4); dst = c0.h_stage; }
        RT_CUDA(cudaMemcpyAsync(dst, c0.d_out, (size_t)W * H * 4, cudaMemcpyDeviceToHost, c0.stream));
        RT_CUDA(cudaStreamSynchronize(c0.stream));
        if (!direct) copy_frame(host32, c0.h_stage, (size_t)W * H * 4);
    }

    if (opt_in.stats) {
        RenderStats& st = *opt_in.stats;
        st = RenderStats{};
        st.grid = (uint32_t)launches[0].grid; st.block = (uint32_t)launches[0].block;
        st.resident   = launches[0].resident ? 1u : 0u;
        st.smem_bytes = st.resident ? (uint32_t)launches[0].hot_bytes : 0u;
        st.filtered   = launches[0].filtered ? 1u : 0u;
        st.culled     = launches[0].culled ? 1u : 0u;
        st.devices    = (uint32_t)N;
        st.peer_gather = peer ? 1u : 0u;
        for (int d = 0; d < N; ++d) {
            if (launches[d].launches == 0) continue;
            RT_CUDA(cudaSetDevice(d));
            DeviceContext& c = *ctxs[d];
            RT_CUDA(cudaMemcpyAsync(c.h_slot, launches[d].slot, sizeof(CounterSlot), cudaMemcpyDeviceToHost, c.stream));
            RT_CUDA(cudaStreamSynchronize(c.stream));
            float ms = 0.f;
            RT_CUDA(cudaEventElapsedTime(&ms, c.ev0, c.ev1));
            st.kernel_ms = std::max(st.kernel_ms, ms);          // devices run concurrently
            st.rays += c.h_slot->rays;
            st.stolen_slots += c.h_slot->stolen;
            st.passes_fused = launches[d].passes_fused;
            st.paths_per_lane = launches[d].paths_per_lane;
            st.launches += launches[d].launches;
            st.sample_items = launches[d].sample_items ? 1u : 0u;
            Options o = base; o.shard_index = (uint32_t)d;
            if (base.samples_per_pixel > 0 && base.max_ray_bounces > 0)
                st.samples += shard_pixels(W, H, o, launches[d].n_tiles) * (uint64_t)base.samples_per_pixel;
        }
        st.total_ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t_begin).count();
    }
}

Framebuffer ray_trace(const World& world, const Camera& camera, Framebuffer framebuffer, Options& options)
{
    if (framebuffer.pixels.size() != framebuffer.width * framebuffer.height)
        framebuffer.pixels.resize(framebuffer.width * framebuffer.height, ColorU8{0, 0, 0, 0});
    Options o     = options;
    o.shard_index = 0;
    o.shard_count = 1;
    o.accum_in = o.accum_out = o.no_resolve = false;
    ray_trace_into(world, camera, framebuffer.width, framebuffer.height, o, framebuffer.pixels.data(), nullptr,
                   nullptr, nullptr);
    return framebuffer;
}

int device_count()
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

double measure_fp32_peak_tflops(int device, float* sm_clock_mhz_out)
{
    std::lock_guard<std::mutex> lock(g_mutex);
    const int dev = resolve_device(device);
    RT_CUDA(cudaSetDevice(dev));
    DeviceContext& ctx = context_for(dev);
    const int block = 256, grid = ctx.num_sms * 8, iters = 16384;
    float* d = nullptr;
    RT_CUDA(cudaMalloc(&d, (size_t)grid * block * sizeof(float)));
    double best = 0.0;
    for (int rep = 0; rep < 5; ++rep) {
        RT_CUDA(cudaEventRecord(ctx.ev0, ctx.stream));
        RT_CUDA(launch_ffma_peak(d, iters, grid, block, ctx.stream));
        RT_CUDA(cudaEventRecord(ctx.ev1, ctx.stream));
        RT_CUDA(cudaStreamSynchronize(ctx.stream));
        float ms = 0.f;
        RT_CUDA(cudaEventElapsedTime(&ms, ctx.ev0, ctx.ev1));
        if (rep > 0) best = std::max(best, ffma_peak_flops_per_launch(iters, grid, block) / (ms * 1e-3) / 1e12);
    }
    RT_CUDA(cudaFree(d));
    if (sm_clock_mhz_out) {
        int khz = 0;
        RT_CUDA(cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, dev));
        *sm_clock_mhz_out = khz / 1000.0f;
    }
    return best;
}

long long selftest_division(int device, unsigned long long operand_sets, uint32_t seed)
{
    std::lock_guard<std::mutex> lock(g_mutex);
    const int dev = resolve_device(device);
    RT_CUDA(cudaSetDevice(dev));
    DeviceContext& ctx = context_for(dev);
    const int block = 256, grid = ctx.num_sms * 4;
    const unsigned long long per_thread = (operand_sets + (unsigned long long)grid * block - 1) / ((unsigned long long)grid * block);
    unsigned long long* d = nullptr;
    RT_CUDA(cudaMalloc(&d, sizeof *d));
    RT_CUDA(cudaMemsetAsync(d, 0, sizeof *d, ctx.stream));
    RT_CUDA(launch_selftest_division(per_thread, seed, grid, block, d, ctx.stream));
    unsigned long long h = 0;
    RT_CUDA(cudaMemcpyAsync(&h, d, sizeof h, cudaMemcpyDeviceToHost, ctx.stream));
    RT_CUDA(cudaStreamSynchronize(ctx.stream));
    RT_CUDA(cudaFree(d));
    return (long long)h;
}

long long selftest_sqrt(int device)
{
    std::lock_guard<std::mutex> lock(g_mutex);
    const int dev = resolve_device(device);
    DeviceGuard guard(dev);
    DeviceContext& ctx = context_for(dev);
    unsigned long long* d = nullptr;
    RT_CUDA(cudaMalloc(&d, sizeof *d));
    RT_CUDA(cudaMemsetAsync(d, 0, sizeof *d, ctx.stream));
    RT_CUDA(launch_selftest_sqrt(ctx.num_sms * 8, 256, d, ctx.stream));
    unsigned long long h = 0;
    RT_CUDA(cudaMemcpyAsync(&h, d, sizeof h, cudaMemcpyDeviceToHost, ctx.stream));
    RT_CUDA(cudaStreamSynchronize(ctx.stream));
    RT_CUDA(cudaFree(d));
    return (long long)h;
}

// ---- device memory helpers for the multi-process peer-store gather (multi.py) ----
void* device_alloc(size_t bytes, int device)
{
    void* p = nullptr;
    if (device < 0) { RT_CUDA(cudaMalloc(&p, bytes)); return p; }
    DeviceGuard guard(resolve_device(device));
    RT_CUDA(cudaMalloc(&p, bytes));
    return p;
}
void device_free(void* p)
{
    if (!p) return;
    cudaPointerAttributes a;
    int cur = -1;
    if (cudaPointerGetAttributes(&a, p) == cudaSuccess && a.type == cudaMemoryTypeDevice &&
        cudaGetDevice(&cur) == cudaSuccess && cur != a.device) {
        cudaSetDevice(a.device);
        cudaFree(p);
        cudaSetDevice(cur);
        return;
    }
    cudaGetLastError();
    cudaFree(p);
}

size_t shard_block_bytes(size_t width, size_t height) { return block_layout(width, height).bytes; }
void   shard_block_init(void* block)
{
    if (!block) throw std::runtime_error("shard_block_init: null block");
    cudaPointerAttributes a;
    RT_CUDA(cudaPointerGetAttributes(&a, block));
    if (a.type != cudaMemoryTypeDevice) throw std::runtime_error("shard_block_init: not device memory");
    DeviceGuard guard(a.device);
    // the whole header is set to the 'queue empty' value; the sums are cleared by every fused-pass frame itself
    RT_CUDA(cudaMemset(block, 0, kBlockHeader));
    const unsigned int v = kQueueExhausted;
    RT_CUDA(cudaMemcpy(block, &v, sizeof v, cudaMemcpyHostToDevice));
}
void ipc_export(const void* device_ptr, unsigned char handle_out[64])
{
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
    cudaIpcMemHandle_t h;
    RT_CUDA(cudaIpcGetMemHandle(&h, const_cast<void*>(device_ptr)));
    std::memcpy(handle_out, &h, 64);
}
void* ipc_open(const unsigned char handle[64])
{
    cudaIpcMemHandle_t h;
    std::memcpy(&h, handle, 64);
    void* p = nullptr;
    RT_CUDA(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
    return p;
}
void ipc_close(void* p) { if (p) RT_CUDA(cudaIpcCloseMemHandle(p)); }
void copy_to_host(void* host_dst, const void* device_src, size_t bytes, void* stream)
{
    RT_CUDA(cudaMemcpyAsync(host_dst, device_src, bytes, cudaMemcpyDeviceToHost, static_cast<cudaStream_t>(stream)));
}

bool is_device_memory(const void* p)
{
    cudaPointerAttributes a;
    cudaError_t e = cudaPointerGetAttributes(&a, p);
    if (e != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeDevice;
}

void* alloc_pinned(size_t bytes)
{
    void* p = nullptr;
    if (cudaMallocHost(&p, bytes) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return p;
}
void free_pinned(void* p) { if (p) cudaFreeHost(p); }

}   // namespace rt
