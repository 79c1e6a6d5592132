"""B200-native render path of the `raytracer` crate — Python host mirror over the C ABI.

The product is `lib/libraytracer.so` (CUDA kernels for sm_100a + C++ host layer, built by
build.py); this module is the thin ctypes binding a Python caller uses.  It mirrors the
reference's own interface for the path, same names and argument meaning:

    reference (raytracer/src/lib.rs)         here
    ----------------------------------------------------------------------
    load_world(source) -> WorldHandle        load_world(source) -> WorldHandle
    render(CFramebuffer, &WorldHandle)       render(framebuffer, handle)
    move_camera_position(camera, x, y, z)    move_camera_position(handle, x, y, z)
    Options::new(spp, depth, ..)             Options(samples_per_pixel, max_ray_bounces, ..)
    ray_trace(world, camera, fb, options)    ray_trace(handle, framebuffer, options)
    image::Framebuffer / write_image         Framebuffer / write_image

There is no CPU fallback anywhere: without the compiled library the import fails, and
without a CUDA device every render call raises RenderError.
"""
from __future__ import annotations

import ctypes as C
import dataclasses
from dataclasses import dataclass
from pathlib import Path
from typing import Optional

import numpy as np

_HERE = Path(__file__).resolve().parent
import os as _os
_variant = _os.environ.get("RT_LIB_VARIANT", "")      # tuning experiments only (build.py)
LIB_PATH = _HERE / ("lib_" + _variant if _variant else "lib") / "libraytracer.so"

SEED_DEFAULT = 2547549            # random.rs:9
OPT_FIXED_JITTER = 0x1
OPT_FAST_MATH = 0x2
OPT_ACCUM_IN = 0x4
OPT_ACCUM_OUT = 0x8
OPT_NO_RESOLVE = 0x10
OPT_FULL_FRAME_OUT = 0x20
OPT_PIXEL_ITEMS = 0x40
OPT_SAMPLE_ITEMS = 0x80
OPT_GROUP_CULL = 0x100
OPT_RESOLVE_EACH_PASS = 0x200
OPT_NO_STEAL = 0x400
OPT_ROW_GATHER = 0x800
DIFFUSE, METAL, DIELECTRIC, EMISSION = 0, 1, 2, 3   # materials.rs:7-12


class RenderError(RuntimeError):
    """A call into libraytracer.so failed (text from rt_last_error())."""


class ParseError(ValueError):
    """load_world rejected the scene text (parser.rs:10-17)."""


class _ColorU8(C.Structure):      # color.rs:3-10
    _fields_ = [("r", C.c_uint8), ("g", C.c_uint8), ("b", C.c_uint8), ("a", C.c_uint8)]


class _CFramebuffer(C.Structure):  # lib.rs:22-27
    _fields_ = [("width", C.c_size_t), ("height", C.c_size_t), ("pixels", C.c_void_p)]


class _WorldHandle(C.Structure):   # lib.rs:29-33
    _fields_ = [("world", C.c_void_p), ("camera", C.c_void_p)]


class RenderStats(C.Structure):
    _fields_ = [("rays", C.c_uint64), ("samples", C.c_uint64), ("kernel_ms", C.c_float),
                ("total_ms", C.c_float), ("launches", C.c_uint32), ("grid", C.c_uint32),
                ("smem_bytes", C.c_uint32), ("resident", C.c_uint32), ("block", C.c_uint32),
                ("devices", C.c_uint32), ("peer_gather", C.c_uint32), ("filtered", C.c_uint32),
                ("sample_items", C.c_uint32), ("culled", C.c_uint32),
                ("passes_fused", C.c_uint32), ("stolen_slots", C.c_uint32),
                ("paths_per_lane", C.c_uint32), ("reserved", C.c_uint32)]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


class PeerQueue(C.Structure):
    """RtPeerQueue: one shard's block (rt_shard_block_bytes) for cross-GPU work stealing."""
    _fields_ = [("block", C.c_void_p), ("shard_index", C.c_uint32), ("reserved", C.c_uint32)]


class _RenderOptions(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("samples_per_pixel", C.c_int32),
                ("max_ray_bounces", C.c_int32), ("seed", C.c_uint32), ("flags", C.c_uint32),
                ("sample_begin", C.c_int32), ("resolve_spp", C.c_int32), ("device", C.c_int32),
                ("tile_rows", C.c_uint32), ("shard_index", C.c_uint32), ("shard_count", C.c_uint32),
                ("n_devices", C.c_uint32), ("stats", C.POINTER(RenderStats)),
                ("passes", C.c_uint32), ("n_peer_queues", C.c_uint32), ("peer_queues", C.POINTER(PeerQueue))]


class AovBuffers(C.Structure):
    """RtAovBuffers: device addresses of the first-hit buffers (0 / None: not written)."""
    _fields_ = [("struct_size", C.c_uint32), ("reserved", C.c_uint32), ("depth", C.c_void_p), ("position", C.c_void_p),
                ("normal", C.c_void_p), ("albedo", C.c_void_p), ("prim", C.c_void_p)]


class _DenoiseOptions(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("iterations", C.c_uint32), ("sigma_color", C.c_float),
                ("sigma_normal", C.c_float), ("sigma_plane", C.c_float), ("device", C.c_int32),
                ("stats", C.POINTER(RenderStats))]


class _RayQueryOptions(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("flags", C.c_uint32), ("device", C.c_int32), ("reserved", C.c_uint32),
                ("stats", C.POINTER(RenderStats))]


_lib: Optional[C.CDLL] = None

# Every symbol include/raytracer.h and include/raytracer_b200.h declare.
EXPORTED_SYMBOLS = (
    "load_world", "render", "move_camera_position", "rt_load_world_ext",
    "rt_last_error", "rt_abi_version", "rt_device_count", "rt_free_world", "rt_free_camera",
    "render_with_options", "rt_render_progressive", "rt_progressive_reset", "rt_render_device", "rt_render_aov_device", "rt_denoise_device",
    "rt_trace_rays_device", "rt_occluded_rays_device", "rt_shard_pixel_count",
    "rt_set_camera_at", "rt_set_camera_vertical_fov", "rt_set_camera_look_at", "rt_set_camera_raw",
    "rt_get_camera",
    "rt_camera_aspect_ratio", "rt_world_new", "rt_world_add_sphere", "rt_world_add_triangle",
    "rt_world_sphere_count", "rt_world_triangle_count", "rt_world_get_sphere", "rt_world_get_triangle",
    "rt_world_to_text", "rt_write_image", "rt_write_image_p6",
    "rt_alloc_pixels", "rt_free_pixels", "rt_measure_fp32_peak", "rt_selftest_division", "rt_selftest_sqrt",
    "rt_device_alloc", "rt_device_free", "rt_shard_block_bytes", "rt_shard_block_init", "rt_ipc_export", "rt_ipc_open", "rt_ipc_close", "rt_copy_to_host",
)


def lib() -> C.CDLL:
    """Load libraytracer.so (fails loudly when the extension has not been built)."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise ImportError(f"{LIB_PATH} is missing: run `python rust-swift-raytracer_b200/build.py` "
                          "(there is no Python/CPU fallback for the render path)")
    L = C.CDLL(str(LIB_PATH))
    f3 = C.POINTER(C.c_float)
    hp = C.POINTER(_WorldHandle)
    L.load_world.restype = hp
    L.load_world.argtypes = [C.c_char_p]
    L.rt_load_world_ext.restype = hp
    L.rt_load_world_ext.argtypes = [C.c_char_p, C.c_uint32]
    L.render.restype = _CFramebuffer
    L.render.argtypes = [_CFramebuffer, hp]
    L.move_camera_position.restype = C.c_void_p
    L.move_camera_position.argtypes = [C.c_void_p, C.c_float, C.c_float, C.c_float]
    L.rt_last_error.restype = C.c_char_p
    L.rt_abi_version.restype = C.c_uint32
    L.rt_device_count.restype = C.c_int
    L.rt_free_world.argtypes = [hp]
    L.rt_free_world.restype = None
    L.rt_free_camera.argtypes = [C.c_void_p]
    L.rt_free_camera.restype = None
    L.render_with_options.restype = _CFramebuffer
    L.render_with_options.argtypes = [_CFramebuffer, hp, C.POINTER(_RenderOptions)]
    L.rt_render_progressive.restype = _CFramebuffer
    L.rt_render_progressive.argtypes = [_CFramebuffer, hp, C.POINTER(_RenderOptions), C.POINTER(C.c_int32)]
    L.rt_progressive_reset.restype = None
    L.rt_progressive_reset.argtypes = [hp]
    L.rt_render_device.restype = C.c_int
    L.rt_render_device.argtypes = [hp, C.POINTER(_RenderOptions), C.c_size_t, C.c_size_t, C.c_void_p,
                                   C.c_void_p, C.c_void_p]
    if not _variant or hasattr(L, "rt_render_aov_device"):
        L.rt_render_aov_device.restype = C.c_int
        L.rt_render_aov_device.argtypes = [hp, C.POINTER(_RenderOptions), C.c_size_t, C.c_size_t, C.POINTER(AovBuffers),
                                           C.c_void_p]
    if not _variant or hasattr(L, "rt_denoise_device"):
        L.rt_denoise_device.restype = C.c_int
        L.rt_denoise_device.argtypes = [C.POINTER(_DenoiseOptions), C.c_size_t, C.c_size_t, C.c_void_p, C.c_int32,
                                        C.POINTER(AovBuffers), C.c_void_p, C.c_void_p, C.c_void_p]
    if not _variant or hasattr(L, "rt_trace_rays_device"):
        L.rt_trace_rays_device.restype = C.c_int
        L.rt_trace_rays_device.argtypes = [hp, C.POINTER(_RayQueryOptions), C.c_size_t, C.c_void_p, C.POINTER(AovBuffers),
                                           C.c_void_p]
    if not _variant or hasattr(L, "rt_occluded_rays_device"):
        L.rt_occluded_rays_device.restype = C.c_int
        L.rt_occluded_rays_device.argtypes = [hp, C.POINTER(_RayQueryOptions), C.c_size_t, C.c_void_p, C.c_void_p,
                                              C.c_void_p]
    L.rt_shard_pixel_count.restype = C.c_size_t
    L.rt_shard_pixel_count.argtypes = [C.c_size_t, C.c_size_t, C.c_uint32, C.c_uint32, C.c_uint32]
    L.rt_set_camera_at.restype = C.c_int
    L.rt_set_camera_at.argtypes = [hp, f3, C.c_float]
    L.rt_set_camera_vertical_fov.restype = C.c_int
    L.rt_set_camera_vertical_fov.argtypes = [hp, f3, C.c_float, C.c_float]
    L.rt_set_camera_look_at.restype = C.c_int
    L.rt_set_camera_look_at.argtypes = [hp, f3, f3, f3, C.c_float, C.c_float]
    L.rt_set_camera_raw.restype = C.c_int
    L.rt_set_camera_raw.argtypes = [hp, f3]
    L.rt_get_camera.restype = None
    L.rt_get_camera.argtypes = [C.c_void_p, f3]
    L.rt_camera_aspect_ratio.restype = C.c_float
    L.rt_camera_aspect_ratio.argtypes = [C.c_void_p]
    L.rt_world_new.restype = hp
    L.rt_world_new.argtypes = [f3, C.c_float]
    L.rt_world_add_sphere.restype = C.c_int
    L.rt_world_add_sphere.argtypes = [hp, f3, C.c_float, C.c_uint32, f3, C.c_float]
    L.rt_world_add_triangle.restype = C.c_int
    L.rt_world_add_triangle.argtypes = [hp, f3, f3, f3, C.c_uint32, f3, C.c_float]
    L.rt_world_sphere_count.restype = C.c_size_t
    L.rt_world_sphere_count.argtypes = [hp]
    L.rt_world_triangle_count.restype = C.c_size_t
    L.rt_world_triangle_count.argtypes = [hp]
    L.rt_world_get_sphere.restype = C.c_int
    L.rt_world_get_sphere.argtypes = [hp, C.c_size_t, f3]
    L.rt_world_get_triangle.restype = C.c_int
    L.rt_world_get_triangle.argtypes = [hp, C.c_size_t, f3]
    L.rt_world_to_text.restype = C.c_size_t
    L.rt_world_to_text.argtypes = [hp, C.c_char_p, C.c_size_t]
    L.rt_write_image.restype = C.c_int
    L.rt_write_image.argtypes = [_CFramebuffer, C.c_char_p]
    L.rt_write_image_p6.restype = C.c_int
    L.rt_write_image_p6.argtypes = [_CFramebuffer, C.c_char_p]
    L.rt_alloc_pixels.restype = C.c_void_p
    L.rt_alloc_pixels.argtypes = [C.c_size_t, C.c_size_t]
    L.rt_free_pixels.restype = None
    L.rt_free_pixels.argtypes = [C.c_void_p]
    L.rt_measure_fp32_peak.restype = C.c_double
    L.rt_measure_fp32_peak.argtypes = [C.c_int]
    L.rt_device_alloc.restype = C.c_void_p
    L.rt_device_alloc.argtypes = [C.c_size_t]
    L.rt_device_free.restype = None
    L.rt_device_free.argtypes = [C.c_void_p]
    if not _variant or hasattr(L, "rt_shard_block_bytes"):      # an A/B build of an older ABI may lack them
        L.rt_shard_block_bytes.restype = C.c_size_t
        L.rt_shard_block_bytes.argtypes = [C.c_size_t, C.c_size_t]
        L.rt_shard_block_init.restype = C.c_int
        L.rt_shard_block_init.argtypes = [C.c_void_p]
    L.rt_ipc_export.restype = C.c_int
    L.rt_ipc_export.argtypes = [C.c_void_p, C.c_char_p]
    L.rt_ipc_open.restype = C.c_void_p
    L.rt_ipc_open.argtypes = [C.c_char_p]
    L.rt_ipc_close.restype = C.c_int
    L.rt_ipc_close.argtypes = [C.c_void_p]
    L.rt_copy_to_host.restype = C.c_int
    L.rt_copy_to_host.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
    if not _variant or hasattr(L, "rt_selftest_sqrt"):
        L.rt_selftest_sqrt.restype = C.c_longlong
        L.rt_selftest_sqrt.argtypes = [C.c_int]
    L.rt_selftest_division.restype = C.c_longlong
    L.rt_selftest_division.argtypes = [C.c_int, C.c_ulonglong, C.c_uint32]
    _lib = L
    return L


def last_error() -> str:
    return lib().rt_last_error().decode("utf-8", "replace")


def device_count() -> int:
    return lib().rt_device_count()


def _f3(v):
    return (C.c_float * 3)(float(v[0]), float(v[1]), float(v[2]))


@dataclass
class Options:
    """common.rs:289-294 `Options` (+ the additive fields of RtRenderOptions)."""
    samples_per_pixel: int = 32          # Options::default(), common.rs:309-316
    max_ray_bounces: int = 8
    seed: int = SEED_DEFAULT
    fixed_jitter: bool = False           # deterministic mode
    fast_math: bool = False
    sample_begin: int = 0
    resolve_spp: int = 0
    device: int = -1
    tile_rows: int = 16
    shard_index: int = 0
    shard_count: int = 1
    accum_in: bool = False
    accum_out: bool = False
    no_resolve: bool = False
    full_frame_out: bool = False         # sharded, but the device buffers are full frames (peer / IPC mapped)
    n_devices: int = 0                   # > 1: this process renders on devices 0..n-1 (render_with_options only)
    sample_items: Optional[bool] = None  # scheduling: None auto, False whole pixels per lane, True single samples
    group_cull: bool = False             # opt-in acceleration: bounding spheres over groups of 8 spheres (same hits)
    passes: int = 1                      # progressive passes of samples_per_pixel/passes, fused into one launch
    resolve_each_pass: bool = False      # fused passes: refresh the RGBA8 frame after every pass
    peer_queues: Optional[list] = None   # [(block address, shard index), ...] of ALL shards: cross-GPU work stealing
    no_steal: bool = False               # with peer_queues: static tile deal only
    row_gather: bool = False             # full_frame_out into ANOTHER GPU's frame: stage locally, last CTA copies 16-byte vectors

    def _c(self, stats: Optional[RenderStats]) -> _RenderOptions:
        flags = ((OPT_FIXED_JITTER if self.fixed_jitter else 0) | (OPT_FAST_MATH if self.fast_math else 0) |
                 (OPT_ACCUM_IN if self.accum_in else 0) | (OPT_ACCUM_OUT if self.accum_out else 0) |
                 (OPT_NO_RESOLVE if self.no_resolve else 0) | (OPT_FULL_FRAME_OUT if self.full_frame_out else 0) | (OPT_GROUP_CULL if self.group_cull else 0) |
                 (OPT_RESOLVE_EACH_PASS if self.resolve_each_pass else 0) | (OPT_NO_STEAL if self.no_steal else 0) |
                 (OPT_ROW_GATHER if self.row_gather else 0) |
                 (0 if self.sample_items is None else OPT_SAMPLE_ITEMS if self.sample_items else OPT_PIXEL_ITEMS))
        o = _RenderOptions(C.sizeof(_RenderOptions), int(self.samples_per_pixel), int(self.max_ray_bounces),
                           int(self.seed) & 0xFFFFFFFF, flags, int(self.sample_begin), int(self.resolve_spp),
                           int(self.device), int(self.tile_rows), int(self.shard_index), int(self.shard_count),
                           int(self.n_devices),
                           C.pointer(stats) if stats is not None else None, int(self.passes), 0, None)
        if self.peer_queues:
            arr = (PeerQueue * len(self.peer_queues))(*[PeerQueue(int(b), int(i), 0) for b, i in self.peer_queues])
            o._keep = arr                     # the array must outlive the call
            o.peer_queues = C.cast(arr, C.POINTER(PeerQueue))
            o.n_peer_queues = len(self.peer_queues)
        return o


class Framebuffer:
    """image.rs:9-36: row-major RGBA8, top row first.  `pinned=True` allocates the pixels with
    rt_alloc_pixels so the frame is DMA'd straight into them."""

    def __init__(self, width: int, height: int, pinned: bool = False):
        self.width, self.height = int(width), int(height)
        self._pinned_ptr = None
        if pinned:
            p = lib().rt_alloc_pixels(self.width, self.height)
            if not p:
                raise RenderError(last_error())
            self._pinned_ptr = p
            buf = (C.c_uint8 * (self.width * self.height * 4)).from_address(p)
            self.pixels = np.frombuffer(buf, dtype=np.uint8).reshape(self.height, self.width, 4)
            self.pixels[...] = 0
        else:
            self.pixels = np.zeros((self.height, self.width, 4), dtype=np.uint8)

    def _c(self) -> _CFramebuffer:
        return _CFramebuffer(self.width, self.height, self.pixels.ctypes.data)

    def __del__(self):
        if getattr(self, "_pinned_ptr", None):
            self.pixels = None
            lib().rt_free_pixels(self._pinned_ptr)
            self._pinned_ptr = None


class WorldHandle:
    """lib.rs:29-33: owns the Rust_WorldHandle* returned by load_world / rt_world_new."""

    def __init__(self, ptr):
        self._ptr = ptr

    @property
    def ptr(self):
        if not self._ptr:
            raise RenderError("world handle already freed")
        return self._ptr

    def free(self):
        if self._ptr:
            lib().rt_free_world(self._ptr)
            self._ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass

    # ---- scene ----
    @property
    def n_spheres(self) -> int:
        return lib().rt_world_sphere_count(self.ptr)

    @property
    def n_triangles(self) -> int:
        return lib().rt_world_triangle_count(self.ptr)

    def sphere(self, index: int) -> np.ndarray:
        """center[3], radius, material type, color[3], param"""
        out = (C.c_float * 9)()
        if lib().rt_world_get_sphere(self.ptr, index, out):
            raise IndexError(index)
        return np.array(out, dtype=np.float32)

    def triangle(self, index: int) -> np.ndarray:
        """v0[3], v1[3], v2[3], normal[3], material type, color[3], param, 0"""
        out = (C.c_float * 18)()
        if lib().rt_world_get_triangle(self.ptr, index, out):
            raise IndexError(index)
        return np.array(out, dtype=np.float32)

    def add_sphere(self, center, radius, material=DIFFUSE, color=(1.0, 1.0, 1.0), param=0.0):
        if lib().rt_world_add_sphere(self.ptr, _f3(center), float(radius), int(material), _f3(color), float(param)):
            raise RenderError(last_error())

    def add_triangle(self, v0, v1, v2, material=DIFFUSE, color=(1.0, 1.0, 1.0), param=0.0):
        if lib().rt_world_add_triangle(self.ptr, _f3(v0), _f3(v1), _f3(v2), int(material), _f3(color), float(param)):
            raise RenderError(last_error())

    def to_text(self) -> str:
        """The world in the reference's text grammar (exact decimal floats; round-trips bit for bit)."""
        n = lib().rt_world_to_text(self.ptr, None, 0)
        if not n:
            raise RenderError(last_error())
        buf = C.create_string_buffer(n)
        lib().rt_world_to_text(self.ptr, buf, n)
        return buf.value.decode("ascii")

    # ---- camera (camera.rs:21-72) ----
    def camera_floats(self) -> np.ndarray:
        out = (C.c_float * 12)()
        lib().rt_get_camera(self.ptr.contents.camera, out)
        return np.array(out, dtype=np.float32)

    def aspect_ratio(self) -> float:
        return lib().rt_camera_aspect_ratio(self.ptr.contents.camera)

    def set_camera_raw(self, camera12):
        """Install origin, lower_left_corner, horizontal, vertical (12 floats) verbatim."""
        a = (C.c_float * 12)(*[float(x) for x in camera12])
        if lib().rt_set_camera_raw(self.ptr, a):
            raise RenderError(last_error())

    def set_camera_at(self, origin, aspect):
        if lib().rt_set_camera_at(self.ptr, _f3(origin), float(aspect)):
            raise RenderError(last_error())

    def set_camera_vertical_fov(self, origin, vfov, aspect):
        if lib().rt_set_camera_vertical_fov(self.ptr, _f3(origin), float(vfov), float(aspect)):
            raise RenderError(last_error())

    def set_camera_look_at(self, origin, look_at, up, vfov, aspect):
        if lib().rt_set_camera_look_at(self.ptr, _f3(origin), _f3(look_at), _f3(up), float(vfov), float(aspect)):
            raise RenderError(last_error())


PARSE_EMISSION = 0x1


def load_world(source, extensions: int = 0) -> WorldHandle:
    """lib.rs:37-46.  Raises ParseError where the reference panics.  extensions=PARSE_EMISSION
    additionally accepts `material NAME : Emission color r g b;` (rt_load_world_ext)."""
    if isinstance(source, str):
        source = source.encode("utf-8")
    p = lib().rt_load_world_ext(source, int(extensions)) if extensions else lib().load_world(source)
    if not p:
        raise ParseError(last_error())
    return WorldHandle(p)


def world_new(camera_origin=(0.0, 0.0, 0.0), aspect_ratio=1.77778) -> WorldHandle:
    """World::new (common.rs:233-235) + Camera::new_at, without the text parser."""
    return WorldHandle(lib().rt_world_new(_f3(camera_origin), float(aspect_ratio)))


def move_camera_position(handle: WorldHandle, x: float, y: float, z: float) -> None:
    """lib.rs:60-63 used the way GameView.swift:200-216 uses it:
    handle.camera = move_camera_position(handle.camera, x, y, z)."""
    h = handle.ptr
    new = lib().move_camera_position(h.contents.camera, float(x), float(y), float(z))
    if not new:
        raise RenderError(last_error())
    h.contents.camera = new


def render(framebuffer: Framebuffer, handle: WorldHandle) -> Framebuffer:
    """lib.rs:49-57: 16 spp, depth 8, into framebuffer.pixels."""
    lib().render(framebuffer._c(), handle.ptr)
    err = last_error()
    if err:
        raise RenderError(err)
    return framebuffer


def render_with_options(framebuffer: Framebuffer, handle: WorldHandle, options: Options,
                        stats: Optional[RenderStats] = None) -> Framebuffer:
    o = options._c(stats)
    lib().render_with_options(framebuffer._c(), handle.ptr, C.byref(o))
    err = last_error()
    if err:
        raise RenderError(err)
    return framebuffer


def render_progressive(framebuffer: Framebuffer, handle: WorldHandle, options: Options,
                       stats: Optional[RenderStats] = None) -> int:
    """rt_render_progressive: adds options.samples_per_pixel samples to the frame accumulated so far
    (restarts when camera / size / world / seed / depth changed).  Returns the total spp in the frame."""
    o = options._c(stats)
    total = C.c_int32(0)
    lib().rt_render_progressive(framebuffer._c(), handle.ptr, C.byref(o), C.byref(total))
    err = last_error()
    if err:
        raise RenderError(err)
    return total.value


def ray_trace(handle: WorldHandle, framebuffer: Framebuffer, options: Options,
              stats: Optional[RenderStats] = None) -> Framebuffer:
    """common.rs:320-361 (world + camera travel together in the handle, as in lib.rs:53-54)."""
    return render_with_options(framebuffer, handle, options, stats)


def render_device(handle: WorldHandle, options: Options, width: int, height: int, device_pixels: int,
                  device_accum: int = 0, stream: int = 0, stats: Optional[RenderStats] = None) -> None:
    """rt_render_device: device_pixels / device_accum / stream are raw addresses
    (e.g. torch.Tensor.data_ptr(), torch.cuda.Stream.cuda_stream)."""
    o = options._c(stats)
    rc = lib().rt_render_device(handle.ptr, C.byref(o), int(width), int(height),
                                C.c_void_p(device_pixels or None), C.c_void_p(device_accum or None),
                                C.c_void_p(stream or None))
    if rc:
        raise RenderError(last_error())


def render_aov_device(handle: WorldHandle, options: Optional[Options], width: int, height: int, depth: int = 0,
                      position: int = 0, normal: int = 0, albedo: int = 0, prim: int = 0, stream: int = 0,
                      stats: Optional[RenderStats] = None) -> None:
    """rt_render_aov_device: World::hit of the camera ray of sample options.sample_begin of every pixel, written to
    whichever buffers are given as raw device addresses (float32 [H][W] depth, [H][W][3] position / normal / albedo,
    int32 [H][W] prim; e.g. torch.Tensor.data_ptr()).  stream: a raw cudaStream_t (torch.cuda.Stream.cuda_stream);
    0 = the library's stream, the call then returns when the buffers are written."""
    o = (options if options is not None else Options())._c(stats)
    b = AovBuffers(C.sizeof(AovBuffers), 0, depth or None, position or None, normal or None, albedo or None, prim or None)
    rc = lib().rt_render_aov_device(handle.ptr, C.byref(o), int(width), int(height), C.byref(b), C.c_void_p(stream or None))
    if rc:
        raise RenderError(last_error())


def render_aov(handle: WorldHandle, width: int, height: int, options: Optional[Options] = None,
               stats: Optional[RenderStats] = None) -> dict:
    """First-hit buffers of a width x height frame as torch tensors on the options' device (the current CUDA device
    when options.device is -1): {"depth": f32 [H,W], "position" / "normal" / "albedo": f32 [H,W,3], "prim": i32 [H,W]}.
    See render_aov_device.  Returns when the buffers are written."""
    import torch                                      # imported here: the package itself needs only numpy
    options = options if options is not None else Options()
    dev = torch.device("cuda", options.device if options.device >= 0 else torch.cuda.current_device())
    H, W = int(height), int(width)
    out = {"depth": torch.empty((H, W), dtype=torch.float32, device=dev),
           "position": torch.empty((H, W, 3), dtype=torch.float32, device=dev),
           "normal": torch.empty((H, W, 3), dtype=torch.float32, device=dev),
           "albedo": torch.empty((H, W, 3), dtype=torch.float32, device=dev),
           "prim": torch.empty((H, W), dtype=torch.int32, device=dev)}
    # the tensors come from torch's allocator on its current stream of `dev`: order the kernel after that stream's work
    # by enqueueing on it (the call then returns once the kernel is enqueued, so wait for the stream afterwards)
    stream = torch.cuda.current_stream(dev)
    render_aov_device(handle, options, W, H, *(out[k].data_ptr() for k in ("depth", "position", "normal", "albedo", "prim")),
                      stream=stream.cuda_stream, stats=stats)
    stream.synchronize()
    return out


# the defaults a 0 field of DenoiseOptions selects (RT_DENOISE_DEFAULT_* in raytracer_b200.h)
DENOISE_DEFAULT_ITERATIONS = 5
DENOISE_DEFAULT_SIGMA_COLOR = 1.0
DENOISE_DEFAULT_SIGMA_NORMAL = 0.25
DENOISE_DEFAULT_SIGMA_PLANE = 0.02


@dataclass
class DenoiseOptions:
    """RtDenoiseOptions: a field left at 0 takes its default (DENOISE_DEFAULT_*)."""
    iterations: int = 0                  # 1..10
    sigma_color: float = 0.0             # finite, > 0
    sigma_normal: float = 0.0
    sigma_plane: float = 0.0             # scene units
    device: int = -1

    def _c(self, stats: Optional[RenderStats]) -> _DenoiseOptions:
        return _DenoiseOptions(C.sizeof(_DenoiseOptions), int(self.iterations), float(self.sigma_color),
                               float(self.sigma_normal), float(self.sigma_plane), int(self.device),
                               C.pointer(stats) if stats is not None else None)


def denoise_device(options: Optional[DenoiseOptions], width: int, height: int, accum: int, spp: int, normal: int,
                   position: int, albedo: int, prim: int, pixels: int = 0, color: int = 0, stream: int = 0,
                   stats: Optional[RenderStats] = None) -> None:
    """rt_denoise_device: the edge-avoiding a-trous filter of the float4 colour sums `accum` (mean = sum / spp),
    guided by the first-hit buffers normal / position / albedo (float32 [H][W][3]) and prim (int32 [H][W]); writes
    RGBA8 `pixels` and / or float4 `color`.  All are raw device addresses (torch.Tensor.data_ptr()); stream: a raw
    cudaStream_t, 0 = the library's stream.  Returns after the outputs are written."""
    o = (options if options is not None else DenoiseOptions())._c(stats)
    g = AovBuffers(C.sizeof(AovBuffers), 0, None, position or None, normal or None, albedo or None, prim or None)
    rc = lib().rt_denoise_device(C.byref(o), int(width), int(height), C.c_void_p(accum or None), int(spp), C.byref(g),
                                 C.c_void_p(pixels or None), C.c_void_p(color or None), C.c_void_p(stream or None))
    if rc:
        raise RenderError(last_error())


def denoise(accum, spp: int, guides: dict, options: Optional[DenoiseOptions] = None,
            stats: Optional[RenderStats] = None) -> dict:
    """Denoise a frame given as torch tensors: accum float32 [H,W,4] colour sums of `spp` samples, guides the dict of
    render_aov ("normal", "position", "albedo": float32 [H,W,3], "prim": int32 [H,W]; "depth" is not read), all on the
    same CUDA device.  Returns {"pixels": uint8 [H,W,4], "color": float32 [H,W,4]} on that device."""
    import torch                                      # imported here: the package itself needs only numpy
    H, W = int(accum.shape[0]), int(accum.shape[1])
    dev = accum.device
    want = {"normal": (torch.float32, (H, W, 3)), "position": (torch.float32, (H, W, 3)),
            "albedo": (torch.float32, (H, W, 3)), "prim": (torch.int32, (H, W))}
    if accum.dtype != torch.float32 or tuple(accum.shape) != (H, W, 4) or not accum.is_contiguous():
        raise ValueError("accum must be a contiguous float32 [H, W, 4] tensor")
    for k, (dt, shape) in want.items():
        t = guides[k]
        if t.dtype != dt or tuple(t.shape) != shape or not t.is_contiguous() or t.device != dev:
            raise ValueError(f"guides[{k!r}] must be a contiguous {dt} {list(shape)} tensor on {dev}")
    options = options if options is not None else DenoiseOptions()
    if dev.type != "cuda" or (options.device >= 0 and options.device != dev.index):
        raise ValueError("the tensors must be on the CUDA device the options name")
    o = DenoiseOptions(options.iterations, options.sigma_color, options.sigma_normal, options.sigma_plane, dev.index)
    out = {"pixels": torch.empty((H, W, 4), dtype=torch.uint8, device=dev),
           "color": torch.empty((H, W, 4), dtype=torch.float32, device=dev)}
    # ordered after the work of torch's current stream of `dev`, which made the tensors (returns when written)
    stream = torch.cuda.current_stream(dev)
    denoise_device(o, W, H, accum.data_ptr(), spp, guides["normal"].data_ptr(), guides["position"].data_ptr(),
                   guides["albedo"].data_ptr(), guides["prim"].data_ptr(), out["pixels"].data_ptr(),
                   out["color"].data_ptr(), stream=stream.cuda_stream, stats=stats)
    return out


def render_denoised(handle: WorldHandle, width: int, height: int, options: Optional[Options] = None,
                    denoise_options: Optional[DenoiseOptions] = None) -> dict:
    """Render a frame and denoise it: render_device with RT_OPT_ACCUM_OUT (the colour sums of
    options.samples_per_pixel samples from options.sample_begin), render_aov with fixed jitter at sample 0 (the guides at pixel centres), then
    denoise.  Returns {"pixels": uint8 [H,W,4], "color": float32 [H,W,4]} on the options' device."""
    import torch
    options = options if options is not None else Options()
    dev = torch.device("cuda", options.device if options.device >= 0 else torch.cuda.current_device())
    H, W = int(height), int(width)
    o = dataclasses.replace(options, accum_out=True, accum_in=False, device=dev.index)
    frame = torch.empty((H, W), dtype=torch.int32, device=dev)
    accum = torch.empty((H, W, 4), dtype=torch.float32, device=dev)
    stream = torch.cuda.current_stream(dev)
    render_device(handle, o, W, H, frame.data_ptr(), accum.data_ptr(), stream=stream.cuda_stream)
    guides = render_aov(handle, W, H, Options(seed=options.seed, fixed_jitter=True, sample_begin=0,
                                              group_cull=options.group_cull, device=dev.index))
    return denoise(accum, o.samples_per_pixel, guides, denoise_options)


RAY_OUTPUTS = ("depth", "position", "normal", "albedo", "prim")
_CUDA_STREAM_LEGACY = 0x1                   # cudaStreamLegacy: the legacy default stream as an explicit handle


@dataclass
class RayQueryOptions:
    """RtRayQueryOptions: group_cull sets RT_OPT_GROUP_CULL (the only flag rt_trace_rays_device and
    rt_occluded_rays_device accept; `flags` is OR-ed in verbatim); device -1 = the current device."""
    group_cull: bool = False
    device: int = -1
    flags: int = 0

    def _c(self, stats: Optional[RenderStats]) -> _RayQueryOptions:
        flags = int(self.flags) | (OPT_GROUP_CULL if self.group_cull else 0)
        return _RayQueryOptions(C.sizeof(_RayQueryOptions), flags, int(self.device), 0,
                                C.pointer(stats) if stats is not None else None)


def trace_rays_device(handle: WorldHandle, options: Optional[RayQueryOptions], n: int, rays: int, depth: int = 0,
                      position: int = 0, normal: int = 0, albedo: int = 0, prim: int = 0, stream: int = 0,
                      stats: Optional[RenderStats] = None) -> None:
    """rt_trace_rays_device: World::hit(Ray{o, normalize(direction)}, 0.001, t_max) of n rays, `rays` the raw device
    address of n RtRay records (float32 [n][8]: origin, t_max, direction, reserved; 16-byte aligned), written to
    whichever outputs are given as raw device addresses (float32 [n] depth, [n][3] position / normal / albedo, int32 [n]
    prim).  stream: a raw cudaStream_t, 0 = the library's own non-blocking stream (the call then returns when the
    outputs are written; it does not wait for work on the legacy default stream — pass 1, cudaStreamLegacy, for that).
    An invalid ray is not an error: its prim is -2 (include/raytracer_b200.h has the semantics)."""
    o = (options if options is not None else RayQueryOptions())._c(stats)
    b = AovBuffers(C.sizeof(AovBuffers), 0, depth or None, position or None, normal or None, albedo or None, prim or None)
    rc = lib().rt_trace_rays_device(handle.ptr, C.byref(o), int(n), C.c_void_p(rays or None), C.byref(b),
                                    C.c_void_p(stream or None))
    if rc:
        raise RenderError(last_error())


def _check_rays(origins, directions, device: Optional[int]):
    """The tensor checks of trace_rays and occluded_rays; returns (torch, the rays' device, N)."""
    import torch                                      # imported here: the package itself needs only numpy
    dev = origins.device
    if dev.type != "cuda" or directions.device != dev or (device is not None and device != dev.index):
        raise ValueError("origins and directions must be on one CUDA device (the one `device` names)")
    N = int(origins.shape[0])
    for name, t in (("origins", origins), ("directions", directions)):
        if t.dtype != torch.float32 or tuple(t.shape) != (N, 3):
            raise ValueError(f"{name} must be a float32 [N, 3] tensor")
    return torch, dev, N


def _check_t_max(torch, t_max, N: int, dev) -> None:
    if isinstance(t_max, torch.Tensor) and (t_max.dtype != torch.float32 or tuple(t_max.shape) != (N,) or t_max.device != dev):
        raise ValueError("a t_max tensor must be float32 [N] on the rays' device")


def _query_stream(torch, dev, stream):
    """(s, handle): the stream the rays are packed on and the kernel runs on, and the handle to pass the library."""
    s = stream if stream is not None else torch.cuda.current_stream(dev)
    # The kernel must run after the packing (and after the caller's work that made the inputs), both on s.  A handle
    # of 0 is the legacy default stream, but 0 passed to the library means its own non-blocking stream, which does not
    # wait for the legacy one: name the legacy stream explicitly (cudaStreamLegacy) instead.
    return s, s.cuda_stream or _CUDA_STREAM_LEGACY


def _pack_rays(torch, origins, directions, t_max, N: int, dev):
    """The RtRay records [N, 8] of the rays, on the current stream (the caller makes it the kernel's)."""
    rays = torch.empty((N, 8), dtype=torch.float32, device=dev)
    rays[:, 0:3] = origins
    rays[:, 3] = float("inf") if t_max is None else t_max
    rays[:, 4:7] = directions
    rays[:, 7] = 0.0
    return rays


def trace_rays(handle: WorldHandle, origins, directions, t_max=None, *, cull: bool = False, device: Optional[int] = None,
               stream=None, outputs=RAY_OUTPUTS, stats: Optional[RenderStats] = None) -> dict:
    """Ray queries on torch tensors: origins and directions are CUDA float32 [N, 3] tensors on one device (directions
    need not be normalised); t_max is None (+inf), a float, or a float32 [N] tensor.  Packs the rays into [N, 8] on the
    device and returns {name: tensor} for the names in `outputs` — "depth" f32 [N], "position" / "normal" / "albedo"
    f32 [N, 3], "prim" i32 [N] (-1 a miss, -2 an invalid ray).  stream: None = torch's current stream of the device, and
    the call returns when the outputs are written; a torch.cuda.Stream: the work is enqueued on it and the call returns
    at once.  N == 0 returns empty tensors without a call."""
    torch, dev, N = _check_rays(origins, directions, device)
    unknown = set(outputs) - set(RAY_OUTPUTS)
    if unknown or not outputs:
        raise ValueError(f"outputs must be a non-empty subset of {RAY_OUTPUTS}")
    _check_t_max(torch, t_max, N, dev)
    shapes = {"depth": ((N,), torch.float32), "position": ((N, 3), torch.float32), "normal": ((N, 3), torch.float32),
              "albedo": ((N, 3), torch.float32), "prim": ((N,), torch.int32)}
    s, handle_of_s = _query_stream(torch, dev, stream)
    with torch.cuda.device(dev), torch.cuda.stream(s):   # tensors made and packed in the order of the kernel's stream
        out = {k: torch.empty(shapes[k][0], dtype=shapes[k][1], device=dev) for k in RAY_OUTPUTS if k in outputs}
        if N == 0:
            return out
        rays = _pack_rays(torch, origins, directions, t_max, N, dev)
        addr = {k: (out[k].data_ptr() if k in out else 0) for k in RAY_OUTPUTS}
        trace_rays_device(handle, RayQueryOptions(group_cull=cull, device=dev.index), N, rays.data_ptr(), **addr,
                          stream=handle_of_s, stats=stats)
    if stream is None:
        s.synchronize()
    return out


def occluded_rays_device(handle: WorldHandle, options: Optional[RayQueryOptions], n: int, rays: int, occluded: int,
                         stream: int = 0, stats: Optional[RenderStats] = None) -> None:
    """rt_occluded_rays_device: does World::hit(Ray{o, normalize(direction)}, 0.001, t_max) return a hit, for n rays?
    `rays` is the raw device address of n RtRay records (as for trace_rays_device) and `occluded` that of n bytes:
    1 a hit, 0 none, 2 an invalid ray.  stream: as for trace_rays_device (0 = the library's own non-blocking stream;
    1, cudaStreamLegacy, for the legacy default stream)."""
    o = (options if options is not None else RayQueryOptions())._c(stats)
    rc = lib().rt_occluded_rays_device(handle.ptr, C.byref(o), int(n), C.c_void_p(rays or None),
                                       C.c_void_p(occluded or None), C.c_void_p(stream or None))
    if rc:
        raise RenderError(last_error())


def occluded_rays(handle: WorldHandle, origins, directions, t_max=None, *, cull: bool = False,
                  device: Optional[int] = None, stream=None, stats: Optional[RenderStats] = None):
    """Occlusion queries on torch tensors: the rays of trace_rays (origins and directions CUDA float32 [N, 3], t_max
    None = +inf, a float or a float32 [N] tensor), packed the same way on the same stream.  Returns a torch.uint8 [N]:
    1 where World::hit returns a hit within t_max (a shadow ray to a light at distance t_max is blocked), 0 where it
    returns none, 2 for an invalid ray.  stream as for trace_rays.  N == 0 returns an empty tensor without a call."""
    torch, dev, N = _check_rays(origins, directions, device)
    _check_t_max(torch, t_max, N, dev)
    s, handle_of_s = _query_stream(torch, dev, stream)
    with torch.cuda.device(dev), torch.cuda.stream(s):   # made and packed in the order of the kernel's stream
        out = torch.empty((N,), dtype=torch.uint8, device=dev)
        if N == 0:
            return out
        rays = _pack_rays(torch, origins, directions, t_max, N, dev)
        occluded_rays_device(handle, RayQueryOptions(group_cull=cull, device=dev.index), N, rays.data_ptr(),
                             out.data_ptr(), stream=handle_of_s, stats=stats)
    if stream is None:
        s.synchronize()
    return out


def shard_pixel_count(width: int, height: int, tile_rows: int, shard_index: int, shard_count: int) -> int:
    return lib().rt_shard_pixel_count(width, height, tile_rows, shard_index, shard_count)


def write_image(framebuffer: Framebuffer, path: str, binary: bool = False) -> None:
    """image.rs:59-81 (ASCII P3); binary=True writes P6."""
    f = lib().rt_write_image_p6 if binary else lib().rt_write_image
    if f(framebuffer._c(), str(path).encode()):
        raise OSError(last_error())


def measure_fp32_peak(device: int = -1) -> float:
    v = lib().rt_measure_fp32_peak(device)
    if v < 0:
        raise RenderError(last_error())
    return v


def device_alloc(nbytes: int) -> int:
    p = lib().rt_device_alloc(int(nbytes))
    if not p:
        raise RenderError(last_error())
    return p


def device_free(ptr: int) -> None:
    lib().rt_device_free(C.c_void_p(ptr))


def shard_block_bytes(width: int, height: int) -> int:
    return lib().rt_shard_block_bytes(int(width), int(height))


def shard_block_init(ptr: int) -> None:
    if lib().rt_shard_block_init(C.c_void_p(ptr)):
        raise RenderError(last_error())


def ipc_export(ptr: int) -> bytes:
    buf = C.create_string_buffer(64)
    if lib().rt_ipc_export(C.c_void_p(ptr), buf):
        raise RenderError(last_error())
    return buf.raw


def ipc_open(handle: bytes) -> int:
    p = lib().rt_ipc_open(C.create_string_buffer(handle, 64))
    if not p:
        raise RenderError(last_error())
    return p


def ipc_close(ptr: int) -> None:
    if lib().rt_ipc_close(C.c_void_p(ptr)):
        raise RenderError(last_error())


def copy_to_host(host_ptr: int, device_ptr: int, nbytes: int, stream: int = 0) -> None:
    if lib().rt_copy_to_host(C.c_void_p(host_ptr), C.c_void_p(device_ptr), int(nbytes), C.c_void_p(stream or None)):
        raise RenderError(last_error())


def selftest_division(operand_sets: int = 1 << 28, seed: int = 1, device: int = -1) -> int:
    """Mismatches between the exact kernel's shared-reciprocal divide and the IEEE divide."""
    v = lib().rt_selftest_division(device, int(operand_sets), int(seed) & 0xFFFFFFFF)
    if v < 0:
        raise RenderError(last_error())
    return v


def selftest_sqrt(device: int = -1) -> int:
    """Mismatches between the exact kernel's range-guarded square root and sqrtf over every float bit pattern."""
    v = lib().rt_selftest_sqrt(device)
    if v < 0:
        raise RenderError(last_error())
    return v


# ---- shard geometry shared by the multi-GPU plumbing (tile t belongs to rank t % N) ----

def shard_tile(shard_index: int, shard_count: int, j: int) -> int:
    """rt_shard_tile (rt_types.h): stripes of shard_count tiles are dealt alternately forwards and
    backwards, so that a vertical cost gradient of the frame cancels between the shards."""
    return j * shard_count + ((shard_count - 1 - shard_index) if (j & 1) else shard_index)


def shard_tiles(height: int, tile_rows: int, shard_index: int, shard_count: int):
    """Image-row ranges [(r0, r1), ...] of the tiles shard `shard_index` renders, in the order
    they are packed in its compact buffer."""
    n_tiles = (height + tile_rows - 1) // tile_rows
    out, j = [], 0
    while True:
        t = shard_tile(shard_index, shard_count, j)
        if t >= n_tiles:
            # a later stripe cannot contain a tile either: stripes are whole multiples of shard_count
            return out
        out.append((t * tile_rows, min((t + 1) * tile_rows, height)))
        j += 1
