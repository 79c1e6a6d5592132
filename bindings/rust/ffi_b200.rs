//! ffi_b200.rs — Rust binding of `libraytracer.so`, the B200-native render path.
//!
//! Drop this file into `raytracer/src/` and apply `reference.patch` (same directory): the crate keeps its
//! public Rust API — `raytracer::{load_world, render, move_camera_position, CFramebuffer}` as used by
//! `examples/c_raytracer.rs:7-11`, `common::ray_trace` as used by `src/main.rs:95` — and forwards to the
//! C ABI declared in `include/raytracer.h` / `include/raytracer_b200.h` of the B200 repository.
//!
//! NOT COMPILED in the authoring environment (no rustc/cargo there); every declaration below mirrors the
//! C header field for field, and the C header is exercised by a C caller in the test-suite.
#![allow(non_camel_case_types, dead_code)]

use crate::color::ColorU8;
use std::ffi::CStr;
use std::os::raw::{c_char, c_int, c_void};
use std::ptr::NonNull;

/// `Rust_CFramebuffer` (raytracer.h:22-26) — the crate's own `CFramebuffer` (lib.rs:22-27) has this layout
/// (`NonNull<T>` is ABI-identical to `*mut T`), so lib.rs keeps its type and passes it straight through.
#[repr(C)]
pub struct CFramebuffer {
    pub width: usize,
    pub height: usize,
    pub pixels: NonNull<ColorU8>,
}

/// `Rust_WorldHandle` (raytracer.h:12-15): two pointers; C callers read both and overwrite `camera`.
#[repr(C)]
pub struct WorldHandle {
    pub world: *mut c_void,
    pub camera: *mut c_void,
}

/// `RtRenderStats` (raytracer_b200.h), ABI version 2.
#[repr(C)]
#[derive(Default, Clone, Copy, Debug)]
pub struct RtRenderStats {
    pub rays: u64,
    pub samples: u64,
    pub kernel_ms: f32,
    pub total_ms: f32,
    pub launches: u32,
    pub grid: u32,
    pub smem_bytes: u32,
    pub resident: u32,
    pub block: u32,
    pub devices: u32,
    pub peer_gather: u32,
    pub filtered: u32,
    pub sample_items: u32,
    pub culled: u32,
    pub passes_fused: u32,
    pub stolen_slots: u32,
    pub paths_per_lane: u32,
    pub reserved: u32,
}

#[repr(C)]
pub struct RtPeerQueue {
    pub block: *mut c_void,
    pub shard_index: u32,
    pub reserved: u32,
}

/// `RtRenderOptions` (raytracer_b200.h), ABI version 2.  Zero everything, then set `struct_size`.
#[repr(C)]
pub struct RtRenderOptions {
    pub struct_size: u32,
    pub samples_per_pixel: i32, // common.rs:290
    pub max_ray_bounces: i32,   // common.rs:291
    pub seed: u32,              // 0 -> 2547549 (random.rs:9)
    pub flags: u32,
    pub sample_begin: i32,
    pub resolve_spp: i32,
    pub device: i32,
    pub tile_rows: u32,
    pub shard_index: u32,
    pub shard_count: u32,
    pub n_devices: u32,
    pub stats: *mut RtRenderStats,
    pub passes: u32,
    pub n_peer_queues: u32,
    pub peer_queues: *const RtPeerQueue,
}

impl RtRenderOptions {
    /// `Options::new(samples_per_pixel, max_ray_bounces, ..)` (common.rs:296-308) on the current device.
    pub fn new(samples_per_pixel: i32, max_ray_bounces: i32) -> Self {
        RtRenderOptions {
            struct_size: std::mem::size_of::<RtRenderOptions>() as u32,
            samples_per_pixel,
            max_ray_bounces,
            seed: 0,
            flags: 0,
            sample_begin: 0,
            resolve_spp: 0,
            device: -1,
            tile_rows: 0,
            shard_index: 0,
            shard_count: 0,
            n_devices: 0,
            stats: std::ptr::null_mut(),
            passes: 0,
            n_peer_queues: 0,
            peer_queues: std::ptr::null(),
        }
    }
}

/// `RtAovBuffers` (raytracer_b200.h): device addresses of the first-hit buffers of `rt_render_aov_device`, null = not
/// written.  f32 [H][W] depth, f32 [H][W][3] position / normal / albedo, i32 [H][W] prim; top row first.
#[repr(C)]
pub struct RtAovBuffers {
    pub struct_size: u32, // size_of::<RtAovBuffers>()
    pub reserved: u32,
    pub depth: *mut f32,
    pub position: *mut f32,
    pub normal: *mut f32,
    pub albedo: *mut f32,
    pub prim: *mut i32,
}

/// `RtDenoiseOptions` (raytracer_b200.h): zero-initialise and set struct_size; a field left at 0 takes its default
/// (5 iterations, sigma_color 1.0, sigma_normal 0.25, sigma_plane 0.02).  device -1 = the current device.
#[repr(C)]
pub struct RtDenoiseOptions {
    pub struct_size: u32, // size_of::<RtDenoiseOptions>()
    pub iterations: u32,  // 1..10
    pub sigma_color: f32,
    pub sigma_normal: f32,
    pub sigma_plane: f32,
    pub device: i32,
    pub stats: *mut RtRenderStats,
}

/// `RtTemporalOptions` (raytracer_b200.h): zero-initialise and set struct_size; a field left at 0 takes its default
/// (max_history 8, normal_cos 0.9, plane_tol 0.02).  device -1 = the current device.
#[repr(C)]
pub struct RtTemporalOptions {
    pub struct_size: u32, // size_of::<RtTemporalOptions>()
    pub max_history: u32, // 1..2^20 samples
    pub normal_cos: f32,
    pub plane_tol: f32,
    pub device: i32,
    pub reserved: u32,
    pub stats: *mut RtRenderStats,
}

/// `RtTemporalHistory` (raytracer_b200.h): the previous frame of `rt_temporal_accumulate_device`, every pointer
/// required; pass a null `*const RtTemporalHistory` for no history.
#[repr(C)]
pub struct RtTemporalHistory {
    pub struct_size: u32, // size_of::<RtTemporalHistory>()
    pub reserved: u32,
    pub camera12: *const f32,
    pub guides: *const RtAovBuffers,
    pub color: *const c_void,
    pub length: *const f32,
}

/// `RtSvgfOptions` (raytracer_b200.h): zero-initialise and set struct_size; a field left at 0 takes its default
/// (iterations 5, max_history 8, normal_cos 0.9, plane_tol 0.02, sigma_luminance 0.5, sigma_normal 0.25,
/// sigma_plane 0.02).  device -1 = the current device.
#[repr(C)]
pub struct RtSvgfOptions {
    pub struct_size: u32, // size_of::<RtSvgfOptions>()
    pub iterations: u32,  // 1..10
    pub max_history: u32, // 1..2^20 samples
    pub normal_cos: f32,
    pub plane_tol: f32,
    pub sigma_luminance: f32,
    pub sigma_normal: f32,
    pub sigma_plane: f32,
    pub device: i32,
    pub reserved: u32,
    pub stats: *mut RtRenderStats,
}

/// `RtSvgfHistory` (raytracer_b200.h): the previous frame of `rt_svgf_device`, every pointer required; pass a null
/// `*const RtSvgfHistory` for no history.
#[repr(C)]
pub struct RtSvgfHistory {
    pub struct_size: u32, // size_of::<RtSvgfHistory>()
    pub reserved: u32,
    pub camera12: *const f32,
    pub guides: *const RtAovBuffers,
    pub illum: *const c_void,   // f32x4, the previous call's illum_out
    pub moments: *const c_void, // f32x2, its moments_out
    pub length: *const f32,     // its length_out
}

/// `RtRay` (raytracer_b200.h): one ray of `rt_trace_rays_device`, 32 bytes, the C layout (alignment 4).  The ray
/// BUFFER must start on a 16-byte boundary (the kernel reads each ray as two 16-byte loads); memory from
/// `rt_device_alloc` does.  t_max: sphere hits count when t < t_max, triangle hits when t <= t_max; +inf for an
/// unbounded ray.
#[repr(C)]
pub struct RtRay {
    pub origin: [f32; 3],
    pub t_max: f32,
    pub direction: [f32; 3], // need not be normalised
    pub reserved: f32,
}

/// `RtRayQueryOptions` (raytracer_b200.h): zero-initialise and set struct_size.  flags: 0 or RT_OPT_GROUP_CULL;
/// device -1 = the current device.
#[repr(C)]
pub struct RtRayQueryOptions {
    pub struct_size: u32, // size_of::<RtRayQueryOptions>()
    pub flags: u32,
    pub device: i32,
    pub reserved: u32,
    pub stats: *mut RtRenderStats,
}

pub const RT_OPT_FIXED_JITTER: u32 = 0x1;
pub const RT_OPT_FAST_MATH: u32 = 0x2;
pub const RT_OPT_GROUP_CULL: u32 = 0x100;
pub const RT_MATERIAL_DIFFUSE: u32 = 0; // materials.rs:8
pub const RT_MATERIAL_METAL: u32 = 1; // materials.rs:9
pub const RT_MATERIAL_DIELECTRIC: u32 = 2; // materials.rs:10
pub const RT_MATERIAL_EMISSION: u32 = 3; // materials.rs:11

#[link(name = "raytracer", kind = "dylib")]
extern "C" {
    // ---- the reference's own three exports (raytracer.h:42-47) ----
    /// replaces lib.rs:37-46; NULL + rt_last_error() where the reference panics
    pub fn load_world(source: *const c_char) -> *mut WorldHandle;
    /// replaces lib.rs:49-57: 16 spp, depth 8; the frame is written into `framebuffer.pixels`
    pub fn render(framebuffer: CFramebuffer, handle: *const WorldHandle) -> CFramebuffer;
    /// replaces lib.rs:60-63: consumes `camera`, returns the moved `Camera::new_at` camera
    pub fn move_camera_position(camera: *mut c_void, x: f32, y: f32, z: f32) -> *mut c_void;

    // ---- additive (raytracer_b200.h) ----
    pub fn render_with_options(framebuffer: CFramebuffer, handle: *const WorldHandle,
                               options: *const RtRenderOptions) -> CFramebuffer;
    pub fn rt_last_error() -> *const c_char;
    pub fn rt_free_world(handle: *mut WorldHandle);
    pub fn rt_world_new(camera_origin: *const f32, aspect_ratio: f32) -> *mut WorldHandle; // World::new, common.rs:233
    pub fn rt_world_add_sphere(handle: *mut WorldHandle, center: *const f32, radius: f32, material: u32,
                               color: *const f32, param: f32) -> c_int; // Sphere, common.rs:54-58
    pub fn rt_world_add_triangle(handle: *mut WorldHandle, v0: *const f32, v1: *const f32, v2: *const f32,
                                 material: u32, color: *const f32, param: f32) -> c_int; // Triangle::new, common.rs:116
    /// World::hit (common.rs:237-258) of the camera ray of sample `options.sample_begin` of every pixel, into device
    /// buffers; `stream` null = the library's stream (returns when written).  0 on success.
    pub fn rt_render_aov_device(handle: *const WorldHandle, options: *const RtRenderOptions, width: usize, height: usize,
                                buffers: *const RtAovBuffers, stream: *mut c_void) -> c_int;
    /// Edge-avoiding a-trous filter of the f32x4 colour sums `accum` (mean = sum / spp), guided by the first-hit buffers
    /// `guides` (normal, position, albedo, prim required); writes RGBA8 `device_pixels` and / or f32x4 `device_color`.
    /// Returns after the outputs are written (also on a caller's `stream`).  0 on success.
    pub fn rt_denoise_device(options: *const RtDenoiseOptions, width: usize, height: usize, accum: *const c_void,
                             spp: i32, guides: *const RtAovBuffers, device_pixels: *mut c_void,
                             device_color: *mut c_void, stream: *mut c_void) -> c_int;
    /// The f32x4 colour sums `accum` (mean = sum / spp) blended with the previous frame's colour history, looked up
    /// where each pixel's surface was in the previous camera (`history` null: none); writes f32x4 `color_out`, f32
    /// `length_out` and optionally RGBA8 `device_pixels`.  `stream` null = the library's stream (returns when written),
    /// else returns once enqueued.  0 on success.
    pub fn rt_temporal_accumulate_device(options: *const RtTemporalOptions, width: usize, height: usize,
                                         accum: *const c_void, spp: i32, guides: *const RtAovBuffers,
                                         camera12: *const f32, history: *const RtTemporalHistory,
                                         color_out: *mut c_void, length_out: *mut f32, device_pixels: *mut c_void,
                                         stream: *mut c_void) -> c_int;
    /// Variance-guided filtering: the f32x4 colour sums `accum` (mean = sum / spp) demodulated by the albedo, blended
    /// with the previous frame's illum and luminance moments (`history` null: none), and a-trous filtered with each
    /// pixel's colour weight set by its luminance variance.  Writes the next call's history (f32x4 `illum_out`, f32x2
    /// `moments_out`, f32 `length_out`) and RGBA8 `device_pixels` and / or f32x4 `device_color`.  Returns after the
    /// outputs are written (also on a caller's `stream`).  0 on success.
    pub fn rt_svgf_device(options: *const RtSvgfOptions, width: usize, height: usize, accum: *const c_void, spp: i32,
                          guides: *const RtAovBuffers, camera12: *const f32, history: *const RtSvgfHistory,
                          illum_out: *mut c_void, moments_out: *mut c_void, length_out: *mut f32,
                          device_pixels: *mut c_void, device_color: *mut c_void, stream: *mut c_void) -> c_int;
    /// World::hit(Ray{o, normalize(direction)}, 0.001, t_max) of `n` device-resident rays, record i into element i of
    /// the non-null `hits` arrays (prim -1 a miss, -2 an invalid ray); `stream` null = the library's stream (returns
    /// when written).  0 on success.
    pub fn rt_trace_rays_device(handle: *const WorldHandle, options: *const RtRayQueryOptions, n: usize,
                                rays: *const RtRay, hits: *const RtAovBuffers, stream: *mut c_void) -> c_int;
    /// Does World::hit(Ray{o, normalize(direction)}, 0.001, t_max) return a hit, for `n` device-resident rays:
    /// occluded[i] = 1 a hit, 0 none, 2 an invalid ray (`n` device bytes); options and `stream` as for
    /// rt_trace_rays_device.  0 on success.
    pub fn rt_occluded_rays_device(handle: *const WorldHandle, options: *const RtRayQueryOptions, n: usize,
                                   rays: *const RtRay, occluded: *mut u8, stream: *mut c_void) -> c_int;
    /// device memory on the current device (null + rt_last_error() on failure) and its release
    pub fn rt_device_alloc(bytes: usize) -> *mut c_void;
    pub fn rt_device_free(device_ptr: *mut c_void);
    /// `rt_copy_to_host`: enqueue a device-to-host copy on `stream` (null: the default stream).  0 on success.
    pub fn rt_copy_to_host(host_dst: *mut c_void, device_src: *const c_void, bytes: usize, stream: *mut c_void) -> c_int;
    /// origin, lower_left_corner, horizontal, vertical (camera.rs:8-15) as 12 floats, installed verbatim
    pub fn rt_set_camera_raw(handle: *mut WorldHandle, camera12: *const f32) -> c_int;
}

/// Text of the last failure of any call on this thread ("" if none).
pub fn last_error() -> String {
    unsafe { CStr::from_ptr(rt_last_error()).to_string_lossy().into_owned() }
}

/// Owner of a handle returned by the library (the reference leaks its `Box<WorldHandle>`, lib.rs:42-45;
/// this one is released with `rt_free_world`).  Derefs to `WorldHandle`, so `&*load_world(..)` in
/// `examples/c_raytracer.rs:55` keeps compiling.
pub struct OwnedWorldHandle(pub NonNull<WorldHandle>);

impl std::ops::Deref for OwnedWorldHandle {
    type Target = WorldHandle;
    fn deref(&self) -> &WorldHandle {
        unsafe { self.0.as_ref() }
    }
}
impl std::ops::DerefMut for OwnedWorldHandle {
    fn deref_mut(&mut self) -> &mut WorldHandle {
        unsafe { self.0.as_mut() }
    }
}
impl Drop for OwnedWorldHandle {
    fn drop(&mut self) {
        unsafe { rt_free_world(self.0.as_ptr()) }
    }
}
// The library serialises its callers with one mutex; a handle may move between threads.
unsafe impl Send for OwnedWorldHandle {}
