"""First-hit buffers (rt_render_aov_device / render_aov): depth, position, normal, albedo and primitive id of the camera
ray of sample `sample_begin` of every pixel — World::hit's record, equal to the CPU reference bit for bit.

The reference is `aov_primary_hits_rows` (tests/aov_host/aov_reference.c): the oracle's own camera ray and
orc_world_hit (oracle/rt_oracle.h) for every pixel.  CPU tests: the boundary's rejections, the reference's known answer,
and the device helper (rt_trace.cuh first_hit) built for the host (tests/aov_host/aov_hostsim.cpp) against the
reference.  GPU tests: the kernel against the reference.

Bit patterns are compared exactly, NaNs included, between two CPU computations.  Between the GPU and the CPU a NaN
(degenerate 1-pixel-wide or -high frames divide by zero, as the reference does) is compared as "NaN": IEEE leaves the
sign and payload of a generated NaN to the hardware, and the GPU's canonical NaN is not x86's.
"""
import ctypes as C
import subprocess
from pathlib import Path

import numpy as np
import pytest

import cases

HERE = Path(__file__).resolve().parent
AOV_HOST = HERE / "aov_host"
NAMES = ("depth", "position", "normal", "albedo", "prim")
_ref_lib = None


def primary_hits(ob, world, camera, width, height, *, seed=None, sample_begin=0, fixed_jitter=False, rows=None):
    """The reference buffers {"depth": f32 [H,W], "position" / "normal" / "albedo": f32 [H,W,3], "prim": i32 [H,W]} of an
    oracle world and camera; rows=(begin, end): only image rows [begin, end) are traced, the rest stays zero."""
    global _ref_lib
    if _ref_lib is None:
        ob.build()                                              # librt_oracle.so, which the reference links
        subprocess.run(["make", "-C", str(AOV_HOST), "build/libaov_reference.so"], check=True, capture_output=True)
        ob.lib()                                                # the worlds passed in are objects of this library
        L = C.CDLL(str(AOV_HOST / "build" / "libaov_reference.so"))
        L.aov_primary_hits_rows.restype = C.c_int
        L.aov_primary_hits_rows.argtypes = [C.c_void_p, C.POINTER(ob.Camera), C.c_size_t, C.c_size_t, C.c_size_t,
                                            C.c_size_t, C.c_uint32, C.c_int32, C.c_int32] + [C.c_void_p] * 5
        _ref_lib = L
    H, W = int(height), int(width)
    out = {"depth": np.zeros((H, W), np.float32), "position": np.zeros((H, W, 3), np.float32),
           "normal": np.zeros((H, W, 3), np.float32), "albedo": np.zeros((H, W, 3), np.float32),
           "prim": np.zeros((H, W), np.int32)}
    r0, r1 = rows if rows is not None else (0, H)
    rc = _ref_lib.aov_primary_hits_rows(world.ptr, C.byref(camera), W, H, r0, r1,
                                        int(ob.SEED_DEFAULT if seed is None else seed) & 0xFFFFFFFF, int(sample_begin),
                                        int(bool(fixed_jitter)), *(out[k].ctypes.data for k in NAMES))
    assert rc == 0
    return out


def _bits(a, canonical_nan=False):
    a = np.ascontiguousarray(a)
    if a.dtype == np.float32:
        b = a.view(np.uint32).copy()
        if canonical_nan:
            b[np.isnan(a)] = 0x7FFFFFFF
        return b
    return a


def assert_same(got: dict, want: dict, canonical_nan=False, rows=None):
    for k in NAMES:
        g, w = np.asarray(got[k]), np.asarray(want[k])
        if rows is not None:
            g, w = g[rows[0]:rows[1]], w[rows[0]:rows[1]]
        gb, wb = _bits(g, canonical_nan), _bits(w, canonical_nan)
        bad = np.argwhere(gb != wb)
        assert bad.size == 0, f"{k}: {len(bad)} values differ, first at {bad[0].tolist()}: {g[tuple(bad[0])]} vs {w[tuple(bad[0])]}"


# ---------------------------------------------------------------------------------------------------------- C ABI

def test_header_declares_the_call_and_the_package_exports_it(rt):
    text = (Path(rt.__file__).resolve().parent.parent / "include" / "raytracer_b200.h").read_text()
    assert "int rt_render_aov_device(" in text and "typedef struct RtAovBuffers" in text
    assert "rt_render_aov_device" in rt.EXPORTED_SYMBOLS
    assert hasattr(rt.lib(), "rt_render_aov_device")
    assert C.sizeof(rt.AovBuffers) == 48 and rt.AovBuffers.prim.offset == 40
    assert rt.lib().rt_abi_version() == 2


REJECTED = [
    ("fast_math", dict(fast_math=True), "RT_OPT_FAST_MATH"),
    ("accum_in", dict(accum_in=True), "RT_OPT_ACCUM_IN"),
    ("accum_out", dict(accum_out=True), "RT_OPT_ACCUM_OUT"),
    ("no_resolve", dict(no_resolve=True), "RT_OPT_NO_RESOLVE"),
    ("resolve_each_pass", dict(resolve_each_pass=True), "RT_OPT_RESOLVE_EACH_PASS"),
    ("full_frame_out", dict(full_frame_out=True), "RT_OPT_FULL_FRAME_OUT"),
    ("row_gather", dict(row_gather=True), "RT_OPT_ROW_GATHER"),
    ("no_steal", dict(no_steal=True), "RT_OPT_NO_STEAL"),
    ("shards", dict(shard_count=2), "shard_count > 1"),
    ("n_devices", dict(n_devices=2), "n_devices > 1"),
    ("passes", dict(passes=2, samples_per_pixel=2), "passes > 1"),
    ("peer_queues", dict(peer_queues=[(0x1000, 0)]), "peer_queues"),
]


def _host_buffers(W, H):
    return {"depth": np.full((H, W), 7.0, np.float32), "position": np.full((H, W, 3), 7.0, np.float32),
            "normal": np.full((H, W, 3), 7.0, np.float32), "albedo": np.full((H, W, 3), 7.0, np.float32),
            "prim": np.full((H, W), 7, np.int32)}


def _call(rt, handle, opt, W, H, bufs, which=NAMES):
    addr = {k: (bufs[k].ctypes.data if k in which else 0) for k in NAMES}
    rt.render_aov_device(handle, opt, W, H, **addr)


def _untouched(bufs):
    return all((b == 7).all() for b in bufs.values())


@pytest.mark.parametrize("name,fields,text", REJECTED, ids=[r[0] for r in REJECTED])
def test_rejected_options_fail_on_the_host(rt, scenes, name, fields, text):
    h = rt.load_world(scenes.example_world())
    bufs = _host_buffers(8, 4)
    with pytest.raises(rt.RenderError) as e:
        _call(rt, h, rt.Options(**fields), 8, 4, bufs)
    assert str(e.value).startswith("render_aov: ") and text in str(e.value), str(e.value)
    assert _untouched(bufs)


@pytest.mark.parametrize("W,H,which,text", [(8, 4, (), "every buffer is NULL"),
                                            (0, 4, NAMES, "at least 1x1"), (8, 0, ("depth",), "at least 1x1"),
                                            (2**30, 4, ("prim",), "framebuffer too large")])
def test_rejected_buffers_and_sizes_fail_on_the_host(rt, scenes, W, H, which, text):
    h = rt.load_world(scenes.example_world())
    bufs = _host_buffers(8, 4)
    with pytest.raises(rt.RenderError) as e:
        _call(rt, h, rt.Options(), W, H, bufs, which)
    assert text in str(e.value), str(e.value)
    assert _untouched(bufs)


def test_null_buffer_block_and_handle(rt, scenes):
    L = rt.lib()
    h = rt.load_world(scenes.example_world())
    o = rt.Options()._c(None)
    assert L.rt_render_aov_device(h.ptr, C.byref(o), 8, 4, None, None) != 0
    assert "buffers is NULL" in rt.last_error()
    b = rt.AovBuffers(C.sizeof(rt.AovBuffers), 0, 0x1000, None, None, None, None)
    assert L.rt_render_aov_device(None, C.byref(o), 8, 4, C.byref(b), None) != 0
    assert "NULL world handle" in rt.last_error()


def test_valid_call_never_falls_back(rt, scenes):
    """Options a caller renders with (spp, depth, tile_rows, scheduling flags) are accepted; with host arrays the call
    fails — without a device because there is none, with one because the arrays are not device memory — and never
    writes a buffer on the CPU."""
    h = rt.load_world(scenes.example_world())
    bufs = _host_buffers(8, 4)
    opt = rt.Options(samples_per_pixel=16, max_ray_bounces=8, tile_rows=8, resolve_spp=3, sample_items=True,
                     fixed_jitter=True, group_cull=True)
    with pytest.raises(rt.RenderError) as e:
        _call(rt, h, opt, 8, 4, bufs)
    want = "no CUDA device available" if rt.device_count() == 0 else "buffer is not device memory of device"
    assert want in str(e.value), str(e.value)
    assert _untouched(bufs)


# --------------------------------------------------------------------------------------------------------- oracle

def test_oracle_known_answer(ob, scenes):
    """world.txt with its new_at camera at 402x226, fixed jitter: column 200, reference row 112 has u = 200.5/401 and
    v = 112.5/225, both exactly 0.5; the ray goes straight down -z and meets the sphere `0 0 -1 radius 0.5` at
    t = 0.5 (SURVEY.md §8c)."""
    cam, world = ob.parse_input(scenes.default_world())
    W, H = 402, 226
    out = primary_hits(ob, world, cam, W, H, fixed_jitter=True)
    r = H - 1 - 112
    idx = [i for i, s in enumerate(world.spheres()) if s.center.tuple() == (0.0, 0.0, -1.0) and s.radius == 0.5]
    assert len(idx) == 1
    assert out["prim"][r, 200] == idx[0]
    assert out["depth"][r, 200] == np.float32(0.5)
    assert tuple(out["position"][r, 200]) == (0.0, 0.0, -0.5)
    assert tuple(out["normal"][r, 200]) == (0.0, 0.0, 1.0)
    m = world.spheres()[idx[0]].material
    assert tuple(out["albedo"][r, 200]) == tuple(np.float32([m.r, m.g, m.b]))
    # misses: +inf, zeros, the sky colour of the ray, -1
    miss = out["prim"] == -1
    assert miss.any() and (~miss).any()
    assert np.isinf(out["depth"][miss]).all() and (out["position"][miss] == 0).all() and (out["normal"][miss] == 0).all()
    assert (out["albedo"][miss][:, 2] == 1.0).all()                  # sky: b = (1-t) + t
    # a band is exactly that band of the frame
    band = primary_hits(ob, world, cam, W, H, fixed_jitter=True, rows=(100, 116))
    assert_same(band, out, rows=(100, 116))


# ---------------------------------------------------------------------------------------- device helper on the host

def _load_hostsim(name):
    subprocess.run(["make", "-C", str(AOV_HOST), "build/" + name], check=True, capture_output=True)
    L = C.CDLL(str(AOV_HOST / "build" / name))
    L.hostsim_primary_hits.restype = C.c_int
    L.hostsim_primary_hits.argtypes = [C.c_char_p, C.POINTER(C.c_float), C.c_uint32, C.c_uint32, C.c_uint32, C.c_int32,
                                       C.c_uint32] + [C.c_void_p] * 5
    return L


@pytest.fixture(scope="module")
def hostsim():
    return _load_hostsim("libaov_hostsim.so")


@pytest.fixture(scope="module")
def hostsim_perturbed():
    return _load_hostsim("libaov_hostsim_perturb.so")


def _hostsim_hits(L, text, cam, W, H, seed, sample_begin, flags):
    out = {"depth": np.zeros((H, W), np.float32), "position": np.zeros((H, W, 3), np.float32),
           "normal": np.zeros((H, W, 3), np.float32), "albedo": np.zeros((H, W, 3), np.float32),
           "prim": np.zeros((H, W), np.int32)}
    cf = cam.floats()
    rc = L.hostsim_primary_hits(text.encode(), cf.ctypes.data_as(C.POINTER(C.c_float)), W, H, seed, sample_begin, flags,
                                *(out[k].ctypes.data for k in NAMES))
    assert rc == 0, rc
    return out


@pytest.mark.parametrize("case", cases.SMALL_CASES, ids=[c[0] for c in cases.SMALL_CASES])
def test_device_helper_on_host_equals_oracle(hostsim, ob, scenes, case):
    name, key, camera, W, H, spp, depth, fixed = case
    cam, world = cases.oracle_scene(ob, scenes, key, camera)
    text = cases.scene_text(scenes, key)
    walks = (0, 0x80000000) + ((0x40000000,) if world.n_spheres >= 64 else ())
    for sample_begin in (0, 5):
        want = primary_hits(ob, world, cam, W, H, sample_begin=sample_begin, fixed_jitter=fixed)
        for walk in walks:
            got = _hostsim_hits(hostsim, text, cam, W, H, ob.SEED_DEFAULT, sample_begin, walk | (1 if fixed else 0))
            assert_same(got, want)


@pytest.mark.parametrize("seed", range(50))
def test_device_helper_on_random_worlds(hostsim, ob, seed):
    text = cases.random_world(seed)
    cam, world = ob.parse_input(text)
    W, H = 40, 28
    want = primary_hits(ob, world, cam, W, H, seed=1000 + seed, sample_begin=seed % 7)
    for walk in (0, 0x80000000, 0x40000000):
        got = _hostsim_hits(hostsim, text, cam, W, H, 1000 + seed, seed % 7, walk)
        assert_same(got, want)


@pytest.mark.parametrize("seed", range(40, 50))
def test_device_helper_with_perturbed_reciprocals(hostsim_perturbed, ob, seed):
    text = cases.random_world(seed, n_spheres=66, n_triangles=40)
    cam, world = ob.parse_input(text)
    W, H = 36, 24
    want = primary_hits(ob, world, cam, W, H)
    for walk in (0, 0x80000000, 0x40000000):
        assert_same(_hostsim_hits(hostsim_perturbed, text, cam, W, H, ob.SEED_DEFAULT, 0, walk), want)


@pytest.mark.parametrize("W,H", [(1, 1), (7, 1), (1, 5)])
def test_device_helper_on_degenerate_frames(hostsim, ob, scenes, W, H):
    cam, world = ob.parse_input(scenes.example_world())
    for fixed in (False, True):
        want = primary_hits(ob, world, cam, W, H, fixed_jitter=fixed)
        assert_same(_hostsim_hits(hostsim, scenes.example_world(), cam, W, H, ob.SEED_DEFAULT, 0, int(fixed)), want)


# ------------------------------------------------------------------------------------------------------------ GPU

def _gpu(gpu_rt, handle, W, H, **opt):
    st = gpu_rt.RenderStats()
    out = gpu_rt.render_aov(handle, W, H, gpu_rt.Options(**opt), st)
    return {k: v.cpu().numpy() for k, v in out.items()}, st


@pytest.mark.gpu
@pytest.mark.parametrize("case", cases.SMALL_CASES, ids=[c[0] for c in cases.SMALL_CASES])
def test_gpu_small_cases(gpu_rt, ob, scenes, case):
    name, key, camera, W, H, spp, depth, fixed = case
    cam, world = cases.oracle_scene(ob, scenes, key, camera)
    h = cases.product_scene(gpu_rt, scenes, key, camera)
    for fixed_jitter in (True, False):
        for sample_begin in (0, 5):
            want = primary_hits(ob, world, cam, W, H, sample_begin=sample_begin, fixed_jitter=fixed_jitter)
            got, st = _gpu(gpu_rt, h, W, H, sample_begin=sample_begin, fixed_jitter=fixed_jitter,
                           samples_per_pixel=spp, max_ray_bounces=depth)
            assert_same(got, want, canonical_nan=True)
            assert st.rays == W * H and st.samples == W * H and st.launches == 1


@pytest.mark.gpu
@pytest.mark.parametrize("W,H", [(1, 1), (7, 1), (1, 5), (123, 77)])
def test_gpu_sizes(gpu_rt, ob, scenes, W, H):
    cam, world = ob.parse_input(scenes.example_world())
    h = gpu_rt.load_world(scenes.example_world())
    for fixed in (False, True):
        got, _ = _gpu(gpu_rt, h, W, H, fixed_jitter=fixed)
        assert_same(got, primary_hits(ob, world, cam, W, H, fixed_jitter=fixed), canonical_nan=True)


@pytest.mark.gpu
def test_gpu_empty_world_is_all_sky(gpu_rt, ob):
    h = gpu_rt.world_new((0.0, 0.0, 0.0), 1.5)
    cam = ob.camera_new_at((0.0, 0.0, 0.0), 1.5)
    got, _ = _gpu(gpu_rt, h, 48, 32)
    want = primary_hits(ob, ob.World(), cam, 48, 32)
    assert (got["prim"] == -1).all() and np.isinf(got["depth"]).all()
    assert_same(got, want, canonical_nan=True)


def _four_material_worlds(gpu_rt, ob, emission_only=False):
    spheres = [((0.0, -100.5, -1.0), 100.0, ob.DIFFUSE, (0.8, 0.8, 0.0), 0.0),
               ((0.0, 0.0, -1.0), 0.5, ob.EMISSION, (0.9, 0.6, 0.3), 0.0),
               ((-1.0, 0.0, -1.0), 0.5, ob.DIELECTRIC, (1.0, 1.0, 1.0), 1.5),
               ((1.0, 0.0, -1.0), 0.5, ob.METAL, (0.8, 0.6, 0.2), 0.3),
               ((0.3, 0.4, -0.7), 0.1, ob.EMISSION, (0.2, 0.7, 1.0), 0.0)]
    h = gpu_rt.world_new((0.0, 0.2, 0.6), 1.6)
    world = ob.World()
    for c, r, kind, col, param in spheres:
        if emission_only:
            kind, param = ob.EMISSION, 0.0
        h.add_sphere(c, r, kind, col, param)
        world.add_sphere(c, r, ob.material(kind, col, param))
    h.add_triangle((-2.0, -0.4, -2.0), (2.0, -0.4, -2.0), (0.0, 1.5, -2.5), ob.EMISSION if emission_only else ob.DIFFUSE,
                   (0.4, 0.5, 0.6))
    world.add_triangle((-2.0, -0.4, -2.0), (2.0, -0.4, -2.0), (0.0, 1.5, -2.5),
                       ob.material(ob.EMISSION if emission_only else ob.DIFFUSE, (0.4, 0.5, 0.6)))
    return h, world, ob.camera_new_at((0.0, 0.2, 0.6), 1.6)


@pytest.mark.gpu
def test_gpu_all_four_materials(gpu_rt, ob):
    h, world, cam = _four_material_worlds(gpu_rt, ob)
    got, _ = _gpu(gpu_rt, h, 160, 100, sample_begin=2)
    assert set(np.unique(got["prim"])) >= {-1, 0, 1, 2, 3, 5}
    assert_same(got, primary_hits(ob, world, cam, 160, 100, sample_begin=2), canonical_nan=True)


@pytest.mark.gpu
@pytest.mark.parametrize("key,W,H,band", [("c3", 1920, 1080, (600, 616)), ("c5", 1280, 720, (400, 416))])
def test_gpu_bands_of_the_large_frames(gpu_rt, ob, scenes, key, W, H, band):
    cam, world = cases.oracle_scene(ob, scenes, key, "file")
    h = cases.product_scene(gpu_rt, scenes, key, "file")
    got, st = _gpu(gpu_rt, h, W, H)
    assert st.filtered == 1 and st.rays == W * H
    assert_same(got, primary_hits(ob, world, cam, W, H, rows=band), canonical_nan=True, rows=band)


@pytest.mark.gpu
def test_gpu_global_memory_path_and_group_cull(gpu_rt, ob, scenes):
    text = scenes.synthetic_world(16000, 0, seed=4242)            # hot lists larger than shared memory
    cam, world = ob.parse_input(text)
    h = gpu_rt.load_world(text)
    W, H = 96, 54
    want = primary_hits(ob, world, cam, W, H)
    got, st = _gpu(gpu_rt, h, W, H)
    assert st.resident == 0 and st.smem_bytes == 0
    assert_same(got, want, canonical_nan=True)
    got, st = _gpu(gpu_rt, h, W, H, group_cull=True)
    assert st.culled == 1
    assert_same(got, want, canonical_nan=True)
    # group cull on a staged world
    cam, world = ob.parse_input(scenes.c3_world())
    h = gpu_rt.load_world(scenes.c3_world())
    got, st = _gpu(gpu_rt, h, W, H, group_cull=True, fixed_jitter=True)
    assert st.culled == 1 and st.resident == 1
    assert_same(got, primary_hits(ob, world, cam, W, H, fixed_jitter=True), canonical_nan=True)


@pytest.mark.gpu
def test_gpu_caller_stream(gpu_rt, ob, scenes):
    import torch
    torch.cuda.set_device(0)
    cam, world = ob.parse_input(scenes.c3_world())
    h = gpu_rt.load_world(scenes.c3_world())
    W, H = 320, 180
    want = primary_hits(ob, world, cam, W, H, sample_begin=1)
    s = torch.cuda.Stream()
    bufs = {"depth": torch.full((H, W), 7.0, device="cuda"), "position": torch.full((H, W, 3), 7.0, device="cuda"),
            "normal": torch.full((H, W, 3), 7.0, device="cuda"), "albedo": torch.full((H, W, 3), 7.0, device="cuda"),
            "prim": torch.full((H, W), 7, dtype=torch.int32, device="cuda")}
    torch.cuda.synchronize()
    with torch.cuda.stream(s):
        torch.cuda._sleep(200_000_000)                              # ~0.1 s of work ahead of the kernel on the stream
    gpu_rt.render_aov_device(h, gpu_rt.Options(sample_begin=1, device=0), W, H,
                             *(bufs[k].data_ptr() for k in NAMES), stream=s.cuda_stream)
    assert not s.query(), "the call waited for the caller's stream"
    assert torch.cuda.current_device() == 0
    s.synchronize()
    assert_same({k: v.cpu().numpy() for k, v in bufs.items()}, want, canonical_nan=True)


@pytest.mark.gpu
@pytest.mark.parametrize("sample_begin", [0, 3])
def test_gpu_albedo_of_an_emission_world_is_its_one_bounce_render(gpu_rt, ob, sample_begin):
    """All materials Emission: one sample of depth 1 is the albedo (hit) or the sky (miss), resolved with
    resolve_spp = 1 — the RGBA8 pack of the albedo buffer (sqrt, x255.999, `as u8`; alpha 2 x 255.999 saturates)."""
    h, _, _ = _four_material_worlds(gpu_rt, ob, emission_only=True)
    W, H = 160, 100
    got, _ = _gpu(gpu_rt, h, W, H, sample_begin=sample_begin, fixed_jitter=True)
    fb = gpu_rt.Framebuffer(W, H)
    gpu_rt.render_with_options(fb, h, gpu_rt.Options(samples_per_pixel=1, max_ray_bounces=1, sample_begin=sample_begin,
                                                     resolve_spp=1, fixed_jitter=True))
    a = got["albedo"].astype(np.float32)
    rgb = np.clip(np.sqrt(a) * np.float32(255.999), 0, 255).astype(np.uint8)
    assert (got["prim"] >= 0).any() and (got["prim"] == -1).any()
    assert np.array_equal(fb.pixels[..., :3], rgb)
    assert (fb.pixels[..., 3] == 255).all()
