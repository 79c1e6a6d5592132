"""Occlusion queries (rt_occluded_rays_device / occluded_rays): does World::hit(Ray{o, normalize(direction)}, 0.001,
t_max) return a hit?  One byte per ray — 1 a hit, 0 none, 2 an invalid ray — under the domain check and normalisation
of the ray queries (include/raytracer_b200.h).

References: the ray-query reference (tests/rays_host/rays_reference.c) mapped through prim >= 0 ? 1 : prim == -1 ? 0 : 2,
and `literal_occluded` below, a literal any-hit restatement over oracle/rt_oracle_np.py: some sphere passes
sphere_hit with the fixed window (0.001, t_max), or some triangle passes triangle_intersect with [0.001, t_max] and has
t < +inf (the mesh's strict minimum starts at +inf).  It validates the proof of DESIGN.md §14 instead of assuming it.
CPU tests: the boundary's rejections, the declaration, known answers, the two references against each other, and the
device function (rt_trace.cuh ray_occluded) built for the host (tests/occlusion_host/occlusion_hostsim.cpp).  GPU
tests: the kernel against the reference and against trace_rays' prim.
"""
import ctypes as C
import subprocess
import zlib
from pathlib import Path

import numpy as np
import pytest

import cases
from test_rays import F, INF, _bounds, _rays, _unit, families, invalid_rays, np_world, npo, reference

HERE = Path(__file__).resolve().parent
ROOT = HERE.parent
OCC_HOST = HERE / "occlusion_host"
SYMBOL = "rt_occluded_rays_device"


def answers(prim):
    """The occlusion answer of a ray-query prim: 1 a hit, 0 a miss, 2 an invalid ray."""
    prim = np.asarray(prim)
    return np.where(prim >= 0, 1, np.where(prim == -1, 0, 2)).astype(np.uint8)


def expected(ob, world, rays):
    return answers(reference(ob, world, rays)["prim"])


def literal_occluded(S, T, ray):
    """One answer, literally: the domain check, NVec3::new, then "does any primitive pass its own test with the initial
    window?" — spheres with (0.001, t_max), the mesh with [0.001, t_max] and its strict minimum's t < +inf."""
    o, t_max, a = tuple(F(x) for x in ray[0:3]), F(ray[3]), tuple(F(x) for x in ray[4:7])
    with np.errstate(all="ignore"):
        s = a[0] * a[0] + a[1] * a[1] + a[2] * a[2]
        valid = all(abs(c) <= F(2.0 ** 40) for c in o) and t_max == t_max and F(2.0 ** -100) <= s <= F(2.0 ** 100)
        if not valid:
            return 2
        d = npo.nvec(*a)
        if any(npo.sphere_hit(sph, o, d, t_max) is not None for sph in S):
            return 1
        for tr in T:
            h = npo.triangle_intersect(tr, o, d, t_max)
            if h is not None and h[0] < F(INF):
                return 1
        return 0


def literal_answers(world, rays):
    S, T = np_world(world)
    return np.array([literal_occluded(S, T, r) for r in np.asarray(rays, np.float32)], np.uint8)


def assert_answers(got, want):
    got, want = np.asarray(got), np.asarray(want)
    bad = np.flatnonzero(got != want)
    assert bad.size == 0, f"{bad.size} of {got.size} answers differ, first at {bad[0]}: {got[bad[0]]} vs {want[bad[0]]}"


# ---------------------------------------------------------------------------------------------------------- C ABI

def test_header_declares_the_call_and_the_package_exports_it(rt, tmp_path):
    text = (ROOT / "include" / "raytracer_b200.h").read_text()
    assert "int rt_occluded_rays_device(" in text
    assert SYMBOL in rt.EXPORTED_SYMBOLS and hasattr(rt.lib(), SYMBOL)
    assert rt.lib().rt_abi_version() == 2
    assert "pub fn rt_occluded_rays_device(" in (ROOT / "bindings" / "rust" / "ffi_b200.rs").read_text()
    # the declaration's exact type, and the layout of what it takes, from a C compiler
    src = tmp_path / "decl.c"
    src.write_text('#include <stddef.h>\n#include <stdint.h>\n#include <stdio.h>\n#include "raytracer_b200.h"\n'
                   "typedef int (*occluded_fn)(const struct Rust_WorldHandle *, const RtRayQueryOptions *, size_t, "
                   "const RtRay *, uint8_t *, void *);\n"
                   "static occluded_fn f;\n"
                   "int main(void) { f = rt_occluded_rays_device; (void)f;\n"
                   "  printf(\"%zu %zu %zu %zu\\n\", sizeof(RtRay), offsetof(RtRay, direction), sizeof(RtRayQueryOptions), "
                   "offsetof(RtRayQueryOptions, stats)); return 0; }\n")
    exe = tmp_path / "decl"
    lib_dir = rt.LIB_PATH.parent
    subprocess.run(["gcc", "-std=c11", "-Wall", "-Werror", "-I", str(ROOT / "include"), str(src), "-o", str(exe),
                    "-L", str(lib_dir), "-lraytracer", f"-Wl,-rpath,{lib_dir}"], check=True)
    got = tuple(map(int, subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()))
    assert got == (32, 16, C.sizeof(rt._RayQueryOptions), rt._RayQueryOptions.stats.offset) == (32, 16, 24, 16)


def _raw_call(rt, handle, n, rays_addr, occluded_addr, options=None, opt_ptr=True):
    o = (options if options is not None else rt.RayQueryOptions())._c(None)
    rc = rt.lib().rt_occluded_rays_device(handle.ptr if handle is not None else None, C.byref(o) if opt_ptr else None,
                                          n, rays_addr, occluded_addr, None)
    return rc, rt.last_error()


def test_rejections_happen_on_the_host_before_any_device_work(rt, scenes):
    h = rt.load_world(scenes.example_world())
    rays = np.zeros((4 + 1, 8), np.float32)                 # one spare record to misalign by
    base = rays.ctypes.data
    aligned = base if base % 16 == 0 else base + (16 - base % 16)
    assert aligned + 4 * 32 <= base + rays.nbytes
    out = np.full(4, 7, np.uint8)
    cases_ = [
        (dict(handle=None), "rt_occluded_rays_device: NULL world handle"),
        (dict(opt_ptr=False), "rt_occluded_rays_device: options is NULL"),
        (dict(options=rt.RayQueryOptions(flags=rt.OPT_FAST_MATH)), "rt_occluded_rays_device: only RT_OPT_GROUP_CULL"),
        (dict(options=rt.RayQueryOptions(flags=rt.OPT_FIXED_JITTER)), "only RT_OPT_GROUP_CULL"),
        (dict(options=rt.RayQueryOptions(flags=0x4)), "only RT_OPT_GROUP_CULL"),
        (dict(options=rt.RayQueryOptions(flags=rt.OPT_GROUP_CULL | 0x200)), "only RT_OPT_GROUP_CULL"),
        (dict(n=0), "occluded_rays: n must be at least 1"),
        (dict(n=2 ** 31), "occluded_rays: n must be at most 2^31 - 1"),
        (dict(rays_addr=None), "occluded_rays: the ray buffer is NULL"),
        (dict(rays_addr=aligned + 4), "occluded_rays: the ray buffer is not 16-byte aligned"),
        (dict(rays_addr=aligned + 8), "not 16-byte aligned"),
        (dict(occluded_addr=None), "occluded_rays: the occluded output is NULL"),
        (dict(occluded_addr=aligned + 4 * 32 - 4), "occluded_rays: the occluded output overlaps the rays"),
        (dict(occluded_addr=aligned - 3), "the occluded output overlaps the rays"),
    ]
    for kw, text in cases_:
        out[:] = 7
        rays[:] = 7.0
        args = dict(handle=h, n=4, rays_addr=aligned, occluded_addr=out.ctypes.data)
        args.update(kw)
        rc, err = _raw_call(rt, **args)
        assert rc != 0 and text in err, (kw, err)
        assert (out == 7).all() and (rays == 7.0).all()


def test_wrong_struct_size_is_rejected(rt, scenes):
    h = rt.load_world(scenes.example_world())
    out = np.full(2, 7, np.uint8)
    rays = np.zeros((2, 8), np.float32)
    for size in (0, 16, 32):
        o = rt._RayQueryOptions(size, 0, -1, 0, None)
        assert rt.lib().rt_occluded_rays_device(h.ptr, C.byref(o), 2, rays.ctypes.data, out.ctypes.data, None) != 0
        assert "rt_occluded_rays_device: options->struct_size must be sizeof(RtRayQueryOptions)" in rt.last_error()
        assert (out == 7).all()


def test_adjacent_output_is_not_an_overlap(rt, scenes):
    h = rt.load_world(scenes.example_world())
    blob = np.full(4096, 7, np.uint8)
    base = blob.ctypes.data + 64 + (-blob.ctypes.data) % 16
    for occ in (base + 8 * 32, base - 8):                     # right after the rays' 256 bytes; ending where they begin
        rc, err = _raw_call(rt, h, 8, base, occ)
        assert rc != 0 and "overlaps" not in err, err
    assert (blob == 7).all()


def test_valid_call_never_falls_back(rt, scenes):
    """A valid call with host arrays fails — without a device because there is none, with one because the arrays are
    not device memory — and never writes an answer on the CPU."""
    h = rt.load_world(scenes.example_world())
    rays = _rays([0.0, 0.0, 0.0], [0.0, 0.0, -1.0])
    assert rays.ctypes.data % 16 == 0
    out = np.full(1, 7, np.uint8)
    for cull in (False, True):
        rc, err = _raw_call(rt, h, 1, rays.ctypes.data, out.ctypes.data, options=rt.RayQueryOptions(group_cull=cull))
        want = "no CUDA device available" if rt.device_count() == 0 else "buffer is not device memory of device"
        assert rc != 0 and want in err, err
        assert (out == 7).all()


def test_python_wrapper_raises_the_library_error(rt, scenes):
    h = rt.load_world(scenes.example_world())
    with pytest.raises(rt.RenderError, match="the occluded output is NULL"):
        rt.occluded_rays_device(h, None, 4, 16, 0)
    with pytest.raises(rt.RenderError, match="n must be at least 1"):
        rt.occluded_rays_device(h, rt.RayQueryOptions(group_cull=True), 0, 16, 64)


# --------------------------------------------------------------------------------------------------- references

def test_known_answers_on_world_txt(ob, scenes):
    """world.txt: the sphere `0 0 -1 r 0.5` lies at t = 0.5 from the origin along (0,0,-1): occluded with t_max = +inf
    and nextafter(0.5, inf), not with t_max = 0.5 (the strict sphere window) or any t_max below."""
    cam, world = ob.parse_input(scenes.default_world())
    assert sum(s.center.tuple() == (0.0, 0.0, -1.0) and s.radius == 0.5 for s in world.spheres()) == 1
    t_maxes = (INF, np.nextafter(F(0.5), F(INF)), 0.5, np.nextafter(F(0.5), F(-INF)), 0.25, 0.001, 0.0, -1.0, -INF)
    rays = np.concatenate([_rays([0.0, 0.0, 0.0], [0.0, 0.0, -1.0], t) for t in t_maxes]
                          + [_rays([0.0, 0.0, 0.0], [0.0, 0.0, -7.0], 0.5), _rays([0.0, 0.0, 0.0], [0.0, 0.0, 0.0])])
    want = np.array([1, 1, 0, 0, 0, 0, 0, 0, 0, 0, 2], np.uint8)
    assert_answers(expected(ob, world, rays), want)
    assert_answers(literal_answers(world, rays), want)


def test_triangle_at_exactly_t_max_occludes(ob):
    world = ob.World()
    world.add_triangle((-1.0, -1.0, -2.0), (1.0, -1.0, -2.0), (0.0, 1.0, -2.0), ob.material(ob.DIFFUSE, (0.2, 0.4, 0.6)))
    t = reference(ob, world, _rays([0.0, 0.0, 0.0], [0.0, 0.0, -1.0]))["depth"][0]
    assert t == F(2.0)
    rays = np.concatenate([_rays([0.0, 0.0, 0.0], [0.0, 0.0, -1.0], x) for x in (t, np.nextafter(t, F(-INF)), INF)])
    assert_answers(expected(ob, world, rays), [1, 0, 1])
    assert_answers(literal_answers(world, rays), [1, 0, 1])


def test_answers_are_the_prim_rule_of_trace_rays():
    assert answers(np.array([-2, -1, 0, 1, 7, 2 ** 30], np.int32)).tolist() == [2, 0, 1, 1, 1, 1]


@pytest.mark.parametrize("case", cases.SMALL_CASES, ids=[c[0] for c in cases.SMALL_CASES])
def test_reference_equals_literal_restatement_on_small_cases(ob, scenes, case):
    name, key, camera, W, H, spp, depth, fixed = case
    cam, world = cases.oracle_scene(ob, scenes, key, camera)
    n = 24 if world.n_spheres + world.n_triangles < 100 else 6
    rays = families(ob, world, cam, seed=3 + (zlib.crc32(name.encode()) & 0xFFFF), n=n)
    if world.n_spheres + world.n_triangles >= 100:
        rays = rays[np.random.default_rng(2).permutation(len(rays))[:160]]
    assert_answers(literal_answers(world, rays), expected(ob, world, rays))


@pytest.mark.parametrize("seed", range(20))
def test_reference_equals_literal_restatement_on_random_worlds(ob, seed):
    cam, world = ob.parse_input(cases.random_world(seed, n_spheres=12, n_triangles=10))
    assert world.n_triangles > 0
    rays = families(ob, world, cam, seed=500 + seed, n=12)
    want = expected(ob, world, rays)
    assert_answers(literal_answers(world, rays), want)
    assert {0, 1, 2} <= set(want.tolist())


# ---------------------------------------------------------------------------------------- device function on the host

def _load_hostsim(name):
    subprocess.run(["make", "-C", str(OCC_HOST), "build/" + name], check=True, capture_output=True)
    L = C.CDLL(str(OCC_HOST / "build" / name))
    L.hostsim_occluded_rays.restype = C.c_int
    L.hostsim_occluded_rays.argtypes = [C.c_char_p, C.c_size_t, C.c_void_p, C.c_uint32, C.c_void_p]
    return L


@pytest.fixture(scope="module")
def hostsim():
    return _load_hostsim("libocclusion_hostsim.so")


@pytest.fixture(scope="module")
def hostsim_perturbed():
    return _load_hostsim("libocclusion_hostsim_perturb.so")


DIRECT, FILTER, CULL = 0, 0x80000000, 0x40000000


def _hostsim(L, text, rays, walk):
    rays = np.ascontiguousarray(rays, np.float32)
    out = np.full(len(rays), 7, np.uint8)
    rc = L.hostsim_occluded_rays(text.encode(), len(rays), rays.ctypes.data, walk, out.ctypes.data)
    assert rc == 0, rc
    return out


def _walks(world):
    return (DIRECT, FILTER) + ((CULL,) if world.n_spheres >= 64 else ())


@pytest.mark.parametrize("case", cases.SMALL_CASES, ids=[c[0] for c in cases.SMALL_CASES])
def test_device_function_on_host_equals_reference(hostsim, ob, scenes, case):
    name, key, camera, W, H, spp, depth, fixed = case
    cam, world = cases.oracle_scene(ob, scenes, key, camera)
    text = cases.scene_text(scenes, key)
    rays = families(ob, world, cam, seed=17 + (zlib.crc32(name.encode()) & 0xFFFF), n=96)
    want = expected(ob, world, rays)
    for walk in _walks(world):
        assert_answers(_hostsim(hostsim, text, rays, walk), want)


@pytest.mark.parametrize("seed", range(50))
def test_device_function_on_random_worlds(hostsim, ob, seed):
    text = cases.random_world(seed)
    cam, world = ob.parse_input(text)
    rays = families(ob, world, cam, seed=2000 + seed, n=48)
    want = expected(ob, world, rays)
    for walk in (DIRECT, FILTER, CULL):
        assert_answers(_hostsim(hostsim, text, rays, walk), want)


@pytest.mark.parametrize("seed", range(40, 50))
def test_device_function_with_perturbed_reciprocals(hostsim_perturbed, ob, seed):
    text = cases.random_world(seed, n_spheres=66, n_triangles=40)
    cam, world = ob.parse_input(text)
    rays = families(ob, world, cam, seed=100 + seed, n=48)
    want = expected(ob, world, rays)
    for walk in (DIRECT, FILTER, CULL):
        assert_answers(_hostsim(hostsim_perturbed, text, rays, walk), want)


def test_device_function_on_invalid_rays(hostsim, ob, scenes):
    for text in (scenes.default_world(), cases.random_world(3)):
        cam, world = ob.parse_input(text)
        rays = invalid_rays()
        want = expected(ob, world, rays)
        assert (want == 2).sum() >= 20 and (want != 2).sum() >= 8
        for walk in _walks(world):
            assert_answers(_hostsim(hostsim, text, rays, walk), want)


def _tiny_origin_rays(world, rng):
    """Origins within 2^-63 of the world's origin (o.o below 2^-126: the CULL walk hands them to the FILTER walk), aimed
    at sphere centres and in random directions, with t_max +inf and just past / short of the reference's hit."""
    tiny = np.array([(1e-25, 0, 0), (0, -3e-22, 1e-30), (2.0 ** -70, 2.0 ** -70, -2.0 ** -70), (1e-38, 0, 0),
                     (-2.0 ** -64, 0, 0), (0, 0, 0)], np.float32)
    o = np.repeat(tiny, 8, axis=0)
    S = world.spheres()
    tgt = np.array([S[i].center.tuple() for i in rng.integers(0, len(S), size=len(o))], np.float32)
    return np.concatenate([_rays(o, tgt - o), _rays(o, _unit(rng, len(o)))])


def test_device_function_on_tiny_origins(hostsim, ob):
    for seed in (5, 6, 7):
        text = cases.random_world(seed, n_spheres=80, n_triangles=12)
        cam, world = ob.parse_input(text)
        rays = _tiny_origin_rays(world, np.random.default_rng(seed))
        base = reference(ob, world, rays)
        hit = base["prim"] >= 0
        assert hit.any()
        short = rays[hit].copy()
        short[:, 3] = np.nextafter(base["depth"][hit], F(-INF))
        rays = np.concatenate([rays, short])
        want = expected(ob, world, rays)
        for walk in (DIRECT, FILTER, CULL):
            assert_answers(_hostsim(hostsim, text, rays, walk), want)


# ------------------------------------------------------------------------------------------------------------ GPU

def _gpu(gpu_rt, handle, rays, cull=False, stats=None):
    import torch
    r = torch.from_numpy(np.ascontiguousarray(rays, np.float32)).cuda()
    out = torch.full((len(rays),), 7, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    gpu_rt.occluded_rays_device(handle, gpu_rt.RayQueryOptions(group_cull=cull), len(rays), r.data_ptr(),
                                out.data_ptr(), stats=stats)
    return out.cpu().numpy()


def _gpu_prim(gpu_rt, handle, rays, cull=False):
    import torch
    r = torch.from_numpy(np.ascontiguousarray(rays, np.float32)).cuda()
    prim = torch.full((len(rays),), 7, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    gpu_rt.trace_rays_device(handle, gpu_rt.RayQueryOptions(group_cull=cull), len(rays), r.data_ptr(), prim=prim.data_ptr())
    return prim.cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("case", cases.SMALL_CASES, ids=[c[0] for c in cases.SMALL_CASES])
def test_gpu_small_cases(gpu_rt, ob, scenes, case):
    name, key, camera, W, H, spp, depth, fixed = case
    cam, world = cases.oracle_scene(ob, scenes, key, camera)
    h = cases.product_scene(gpu_rt, scenes, key, camera)
    rays = families(ob, world, cam, seed=23 + (zlib.crc32(name.encode()) & 0xFFFF), n=256)
    want = expected(ob, world, rays)
    for cull in ((False, True) if world.n_spheres >= 64 else (False,)):
        st = gpu_rt.RenderStats()
        assert_answers(_gpu(gpu_rt, h, rays, cull, st), want)
        assert st.rays == len(rays) and st.samples == len(rays) and st.launches == 1 and st.culled == int(cull)
        assert_answers(answers(_gpu_prim(gpu_rt, h, rays, cull)), want)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 31, 33, 1000, 2 ** 20 + 7])
def test_gpu_sizes(gpu_rt, ob, scenes, n):
    cam, world = ob.parse_input(scenes.example_world())
    h = gpu_rt.load_world(scenes.example_world())
    base = families(ob, world, cam, seed=n % 997, n=64)
    rays = base[np.random.default_rng(n).integers(0, len(base), size=n)]
    got = _gpu(gpu_rt, h, rays)
    assert_answers(got, expected(ob, world, rays))


@pytest.mark.gpu
def test_gpu_empty_world_and_four_materials(gpu_rt, ob):
    import test_aov
    h = gpu_rt.world_new((0.0, 0.0, 0.0), 1.5)
    rays = np.concatenate([_rays([0.0, 0.0, 0.0], _unit(np.random.default_rng(3), 500)), invalid_rays()])
    got = _gpu(gpu_rt, h, rays)
    assert set(np.unique(got)) == {0, 2}
    assert_answers(got, expected(ob, ob.World(), rays))
    h, world, cam = test_aov._four_material_worlds(gpu_rt, ob)
    rays = families(ob, world, cam, seed=6, n=400)
    want = expected(ob, world, rays)
    assert set(np.unique(want)) == {0, 1, 2}
    assert_answers(_gpu(gpu_rt, h, rays), want)


@pytest.mark.gpu
def test_gpu_global_memory_path_filter_and_cull(gpu_rt, ob, scenes):
    text = scenes.synthetic_world(16000, 0, seed=4242)            # hot lists larger than shared memory
    cam, world = ob.parse_input(text)
    h = gpu_rt.load_world(text)
    rng = np.random.default_rng(19)
    rays = np.concatenate([families(ob, world, cam, seed=19, n=128), _tiny_origin_rays(world, rng)])
    want = expected(ob, world, rays)
    for cull in (False, True):
        st = gpu_rt.RenderStats()
        assert_answers(_gpu(gpu_rt, h, rays, cull, st), want)
        assert st.resident == 0 and st.smem_bytes == 0 and st.filtered == 1 and st.culled == int(cull)


def _shadow_rays(gpu_rt, h, world, W, H, rng):
    """Shadow rays from the first-hit positions of a W x H frame towards a point light above the world's bounds, t_max
    the distance to the light; plus incoherent rays from the same points."""
    aov = gpu_rt.render_aov(h, W, H, gpu_rt.Options(fixed_jitter=True))
    pos = aov["position"].cpu().numpy().reshape(-1, 3)[aov["prim"].cpu().numpy().reshape(-1) >= 0]
    lo, hi = _bounds(world)
    light = np.array([(lo[0] + hi[0]) / 2, hi[1] + 0.5 * (hi[1] - lo[1]) + 1.0, (lo[2] + hi[2]) / 2], np.float32)
    to_l = light[None, :] - pos
    shadow = _rays(pos, to_l, np.sqrt((to_l.astype(np.float64) ** 2).sum(1)).astype(np.float32))
    return np.concatenate([shadow, _rays(pos, _unit(rng, len(pos)))])


@pytest.mark.gpu
@pytest.mark.parametrize("key,n", [("c3", 2 ** 18), ("c5", 2 ** 14)])
def test_gpu_large_worlds(gpu_rt, ob, scenes, key, n):
    cam, world = cases.oracle_scene(ob, scenes, key, "file")
    h = cases.product_scene(gpu_rt, scenes, key, "file")
    rng = np.random.default_rng(n + 1)
    lo, hi = _bounds(world)
    o = (lo + rng.uniform(size=(n, 3)) * (hi - lo)).astype(np.float32)
    o[: n // 2] = np.array(cam.origin.tuple(), np.float32)
    rays = _rays(o, _unit(rng, n) * np.exp2(rng.integers(-20, 21, size=(n, 1))).astype(np.float32))
    rays[::7, 3] = rng.uniform(0.0, 5.0, size=len(rays[::7]))
    shadow = _shadow_rays(gpu_rt, h, world, 128, 72, rng)
    rays = np.concatenate([rays, shadow[rng.permutation(len(shadow))[: n // 2]]])
    want = expected(ob, world, rays)
    assert (want == 1).any() and (want == 0).any()
    for cull in (False, True):
        st = gpu_rt.RenderStats()
        assert_answers(_gpu(gpu_rt, h, rays, cull, st), want)
        assert st.filtered == 1 and st.resident == 1 and st.culled == int(cull)
        assert_answers(answers(_gpu_prim(gpu_rt, h, rays, cull)), want)


@pytest.mark.gpu
def test_gpu_caller_stream_and_explicit_device(gpu_rt, ob, scenes):
    import torch
    torch.cuda.set_device(0)
    cam, world = ob.parse_input(scenes.c3_world())
    h = gpu_rt.load_world(scenes.c3_world())
    rays = families(ob, world, cam, seed=37, n=512)
    want = expected(ob, world, rays)
    s = torch.cuda.Stream()
    r = torch.from_numpy(rays).cuda()
    out = torch.full((len(rays),), 7, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    with torch.cuda.stream(s):
        torch.cuda._sleep(200_000_000)                              # ~0.1 s of work ahead of the kernel on the stream
    gpu_rt.occluded_rays_device(h, gpu_rt.RayQueryOptions(device=0), len(rays), r.data_ptr(), out.data_ptr(),
                                stream=s.cuda_stream)
    assert not s.query(), "the call waited for the caller's stream"
    assert torch.cuda.current_device() == 0
    s.synchronize()
    assert_answers(out.cpu().numpy(), want)


@pytest.mark.gpu
def test_gpu_stats(gpu_rt, scenes):
    import torch
    h = gpu_rt.load_world(scenes.c3_world())
    n = 100_000
    o = torch.zeros((n, 3), device="cuda")
    d = torch.randn((n, 3), device="cuda")
    for cull in (False, True):
        st = gpu_rt.RenderStats()
        gpu_rt.occluded_rays(h, o, d, cull=cull, stats=st)
        assert st.rays == n and st.samples == n and st.launches == 1
        assert st.kernel_ms > 0 and st.total_ms >= st.kernel_ms and st.grid >= 1 and st.block in (256, 1024)
        assert st.resident == 1 and st.smem_bytes > 0 and st.filtered == 1 and st.culled == int(cull)


@pytest.mark.gpu
def test_gpu_occluded_rays_tensors(gpu_rt, ob, scenes):
    import torch
    cam, world = ob.parse_input(scenes.default_world())
    h = gpu_rt.load_world(scenes.default_world())
    rays = families(ob, world, cam, seed=43, n=128)
    rays[:, 7] = 0.0                                              # occluded_rays packs reserved = 0
    o = torch.from_numpy(rays[:, 0:3].copy()).cuda()
    d = torch.from_numpy(rays[:, 4:7].copy()).cuda()
    t = torch.from_numpy(rays[:, 3].copy()).cuda()
    got = gpu_rt.occluded_rays(h, o, d, t)
    assert got.dtype == torch.uint8 and tuple(got.shape) == (len(rays),) and got.device == o.device
    assert_answers(got.cpu().numpy(), expected(ob, world, rays))
    for t_max in (None, 0.75):
        r = rays.copy()
        r[:, 3] = INF if t_max is None else t_max
        assert_answers(gpu_rt.occluded_rays(h, o, d, t_max, cull=True, device=0).cpu().numpy(), expected(ob, world, r))
    empty = gpu_rt.occluded_rays(h, o[:0], d[:0])
    assert empty.dtype == torch.uint8 and tuple(empty.shape) == (0,)
    s = torch.cuda.Stream()
    got = gpu_rt.occluded_rays(h, o, d, stream=s)
    s.synchronize()
    assert_answers(got.cpu().numpy(), expected(ob, world, _rays(rays[:, 0:3], rays[:, 4:7])))
    with pytest.raises(ValueError):
        gpu_rt.occluded_rays(h, o, d, t[:-1])


@pytest.mark.gpu
def test_gpu_occluded_rays_waits_for_torch_default_stream(gpu_rt, ob, scenes):
    """occluded_rays with stream=None packs the rays on torch's current stream — here the legacy default stream, behind
    ~0.1 s of work — and its kernel must run after that packing, not on a stream that does not wait for it."""
    import torch
    torch.cuda.set_device(0)
    assert torch.cuda.current_stream().cuda_stream == 0
    cam, world = ob.parse_input(scenes.c3_world())
    h = gpu_rt.load_world(scenes.c3_world())
    rays = families(ob, world, cam, seed=53, n=2048)
    rays[:, 7] = 0.0
    want = expected(ob, world, rays)
    o = torch.from_numpy(rays[:, 0:3].copy()).cuda()
    d = torch.from_numpy(rays[:, 4:7].copy()).cuda()
    t = torch.from_numpy(rays[:, 3].copy()).cuda()
    junk = torch.full((len(rays), 8), float("nan"), device="cuda")   # the block the packed rays will likely reuse
    del junk
    torch.cuda.synchronize()
    torch.cuda._sleep(200_000_000)                                  # ahead of the packing on torch's stream
    assert_answers(gpu_rt.occluded_rays(h, o, d, t).cpu().numpy(), want)
