"""Ray queries (rt_trace_rays_device / trace_rays): World::hit(Ray{o, normalize(direction)}, 0.001, t_max) of
caller-supplied rays, with the domain check, the per-ray t_max rule and the first-hit record of
include/raytracer_b200.h — equal to the CPU reference bit for bit.

References: `rays_reference` (tests/rays_host/rays_reference.c, over the oracle's public API: domain check,
orc_normalize, orc_world_hit with t_max = +inf, then the t_max rule), and `literal_hit` below, a literal restatement of
World::hit(ray, 0.001, T) — the shrinking window of common.rs:237-258 starting at T — over oracle/rt_oracle_np.py's
sphere_hit and triangle_intersect, which validates the t_max rule instead of assuming it.  CPU tests: the boundary's
rejections, the layout, known answers, the two references against each other, and the device function (rt_trace.cuh
ray_hit) built for the host (tests/rays_host/rays_hostsim.cpp).  GPU tests: the kernel against the reference.

Bit patterns are compared exactly, NaNs included, between two CPU computations; between the GPU and the CPU a NaN is
compared as "NaN" (an invalid ray's depth is the same quiet NaN on both, but IEEE leaves generated NaNs to the hardware).
"""
import ctypes as C
import subprocess
import sys
import zlib
from pathlib import Path

import numpy as np
import pytest

import cases

HERE = Path(__file__).resolve().parent
ROOT = HERE.parent
RAYS_HOST = HERE / "rays_host"
NAMES = ("depth", "position", "normal", "albedo", "prim")
F = np.float32
INF = float("inf")
_ref_lib = None

sys.path.insert(0, str(ROOT / "oracle"))
import rt_oracle_np as npo  # noqa: E402


def _empty(n):
    return {"depth": np.zeros(n, np.float32), "position": np.zeros((n, 3), np.float32),
            "normal": np.zeros((n, 3), np.float32), "albedo": np.zeros((n, 3), np.float32),
            "prim": np.zeros(n, np.int32)}


def reference(ob, world, rays):
    """The records of rays (float32 [n, 8]) in an oracle world, by tests/rays_host/rays_reference.c."""
    global _ref_lib
    if _ref_lib is None:
        ob.build()
        subprocess.run(["make", "-C", str(RAYS_HOST), "build/librays_reference.so"], check=True, capture_output=True)
        ob.lib()
        L = C.CDLL(str(RAYS_HOST / "build" / "librays_reference.so"))
        L.rays_reference.restype = C.c_int
        L.rays_reference.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p] + [C.c_void_p] * 5
        _ref_lib = L
    rays = np.ascontiguousarray(rays, np.float32)
    out = _empty(len(rays))
    assert _ref_lib.rays_reference(world.ptr, len(rays), rays.ctypes.data, *(out[k].ctypes.data for k in NAMES)) == 0
    return out


def _bits(a, canonical_nan=False):
    a = np.ascontiguousarray(a)
    if a.dtype == np.float32:
        b = a.view(np.uint32).copy()
        if canonical_nan:
            b[np.isnan(a)] = 0x7FFFFFFF
        return b
    return a


def assert_same(got, want, canonical_nan=False, keys=NAMES):
    for k in keys:
        g, w = np.asarray(got[k]), np.asarray(want[k])
        bad = np.argwhere(_bits(g, canonical_nan) != _bits(w, canonical_nan))
        assert bad.size == 0, f"{k}: {len(bad)} values differ, first at {bad[0].tolist()}: {g[tuple(bad[0])]} vs {w[tuple(bad[0])]}"


# ------------------------------------------------------------------------------------------ literal restatement

def np_world(world):
    """The oracle world as rt_oracle_np's (spheres, triangles) tuples (the stored triangle normals are the oracle's)."""
    def f3(v): return (F(v.x), F(v.y), F(v.z))
    def mat(m): return (int(m.type), (F(m.r), F(m.g), F(m.b)), F(m.param))
    S = [(f3(s.center), F(s.radius), mat(s.material)) for s in world.spheres()]
    T = [(f3(t.v0), f3(t.v1), f3(t.v2), f3(t.normal), mat(t.material)) for t in world.triangles()]
    return S, T


def literal_hit(S, T, ray):
    """One record, literally: the domain check, NVec3::new, then World::hit(ray, 0.001, t_max) — every sphere in list
    order with the window (0.001, closest) starting at closest = t_max, then the mesh with [0.001, closest] and its own
    strict minimum — and the record of the first-hit buffers."""
    o, t_max, a = tuple(F(x) for x in ray[0:3]), F(ray[3]), tuple(F(x) for x in ray[4:7])
    with np.errstate(all="ignore"):
        s = a[0] * a[0] + a[1] * a[1] + a[2] * a[2]
        valid = all(abs(c) <= F(2.0 ** 40) for c in o) and t_max == t_max and F(2.0 ** -100) <= s <= F(2.0 ** 100)
        if not valid:
            return F(np.uint32(0x7FFFFFFF).view(np.float32)), (F(0),) * 3, (F(0),) * 3, (F(0),) * 3, -2
        d = npo.nvec(*a)
        closest, rec = t_max, None
        for i, sph in enumerate(S):
            h = npo.sphere_hit(sph, o, d, closest)
            if h is not None:
                closest, rec = h[0], (h[0], h[1], h[2], sph[2], i)
        best, mesh = F(INF), None
        for j, tr in enumerate(T):
            h = npo.triangle_intersect(tr, o, d, closest)
            if h is not None and h[0] < best:
                best, mesh = h[0], (h[0], h[1], tr[3], tr[4], len(S) + j)
        if mesh is not None:
            rec = mesh
        if rec is None:
            st = F(0.5) * (npo.nvec(*d)[1] + F(1.0))
            mt = F(1.0) - st
            sky = (F(1.0) * mt + F(0.5) * st, F(1.0) * mt + F(0.7) * st, F(1.0) * mt + F(1.0) * st)
            return F(INF), (F(0),) * 3, (F(0),) * 3, sky, -1
        t, pos, nrm, m, prim = rec
        alb = (F(1), F(1), F(1)) if m[0] == npo.DIELECTRIC else m[1]
        return t, pos, nrm, alb, prim


def literal_records(world, rays):
    S, T = np_world(world)
    out = _empty(len(rays))
    for i, r in enumerate(np.asarray(rays, np.float32)):
        t, pos, nrm, alb, prim = literal_hit(S, T, r)
        out["depth"][i], out["position"][i], out["normal"][i], out["albedo"][i], out["prim"][i] = t, pos, nrm, alb, prim
    return out


# ------------------------------------------------------------------------------------------------- ray families

def _rays(o, d, t_max=INF):
    o, d = np.asarray(o, np.float32).reshape(-1, 3), np.asarray(d, np.float32).reshape(-1, 3)
    n = max(len(o), len(d))
    r = np.zeros((n, 8), np.float32)
    r[:, 0:3], r[:, 4:7] = o, d
    r[:, 3] = t_max
    return r


def _unit(rng, n):
    v = rng.normal(size=(n, 3))
    return (v / np.linalg.norm(v, axis=1, keepdims=True)).astype(np.float32)


def _bounds(world):
    pts = [s.center.tuple() for s in world.spheres()] + [p.tuple() for t in world.triangles() for p in (t.v0, t.v1, t.v2)]
    pts = np.array(pts or [(0.0, 0.0, 0.0)], np.float64)
    pts = pts[np.all(np.isfinite(pts), axis=1) & np.all(np.abs(pts) < 1e6, axis=1)]
    if not len(pts):
        pts = np.zeros((1, 3))
    return pts.min(0), pts.max(0)


def invalid_rays():
    """Every way a ray can leave the domain, plus the valid rays just inside each bound."""
    big, nxt = F(2.0 ** 40), np.nextafter(F(2.0 ** 40), F(INF))
    good = [0.0, 0.2, 1.0, 1.0, 0.0, 0.0, -1.0, 0.0]
    rays = []
    for k in (0, 1, 2, 3, 4, 5, 6):                       # NaN / +-inf in each field (t_max: only NaN is invalid)
        for v in (np.nan, INF, -INF):
            r = list(good)
            r[k] = v
            rays.append(r)
    for k in (0, 1, 2):                                   # |o.c| = 2^40 (valid) and the next float above (invalid)
        for v in (big, -big, nxt, -nxt):
            r = list(good)
            r[k] = v
            rays.append(r)
    lo, hi = F(2.0 ** -50), F(2.0 ** 50)                  # s = 2^-100 and 2^100 exactly: valid
    for v in (lo, hi, np.nextafter(lo, F(0)), np.nextafter(hi, F(INF)), F(0.0), F(2.0 ** -80), F(2.0 ** 70)):
        rays.append([0.0, 0.0, 0.0, INF, 0.0, 0.0, -v, 0.0])
    # s in range only through the sum (components below 2^-50 each) and s overflowing through the sum
    rays.append([0.0, 0.0, 0.0, INF, F(2.0 ** -51), F(2.0 ** -51), -F(2.0 ** -51), 0.0])
    rays.append([0.0, 0.0, 0.0, INF, F(2.0 ** 49.9), F(2.0 ** 49.9), -F(2.0 ** 49.9), 0.0])
    rays.append([0.0, 0.0, 0.0, INF, 0.0, 0.0, 0.0, 0.0])
    rays.append([0.0, 0.0, 0.0, INF, 0.0, 0.0, -1.0, np.nan])   # `reserved` is ignored
    return np.array(rays, np.float32)


def families(ob, world, cam, seed, n=64):
    """The seeded ray families of a world (float32 [m, 8]); `n` scales the random ones."""
    rng = np.random.default_rng(seed)
    lo, hi = _bounds(world)
    span = np.maximum(hi - lo, 1.0)
    parts = []
    # random origins inside and outside the bounds, directions uniform on the sphere scaled by 2^k, k in [-45, 45]
    o = (lo - 0.5 * span + rng.uniform(size=(n, 3)) * 2.0 * span).astype(np.float32)
    k = rng.integers(-45, 46, size=(n, 1))
    parts.append(_rays(o, _unit(rng, n) * np.exp2(k).astype(np.float32)))
    # secondary-like rays from the first-hit points of camera rays: reflected and random directions
    u, v = rng.uniform(size=n).astype(np.float32), rng.uniform(size=n).astype(np.float32)
    cr = np.array([_camera_vector(cam, uu, vv) for uu, vv in zip(u, v)], np.float32)
    first = reference(ob, world, _rays(np.array(cam.origin.tuple(), np.float32), cr))
    hit = first["prim"] >= 0
    if hit.any():
        p, nn = first["position"][hit], first["normal"][hit]
        d = cr[hit] / np.linalg.norm(cr[hit], axis=1, keepdims=True)
        refl = d - 2.0 * np.sum(d * nn, axis=1, keepdims=True) * nn
        parts += [_rays(p, refl.astype(np.float32)), _rays(p, _unit(rng, len(p)))]
    S, T = world.spheres(), world.triangles()
    if S:
        idx = rng.integers(0, len(S), size=min(n, 4 * len(S)))
        c = np.array([S[i].center.tuple() for i in idx], np.float32)
        r = np.array([abs(S[i].radius) for i in idx], np.float32)[:, None]
        # origins inside spheres; rays aimed at sphere centres; tangent and grazing rays
        parts.append(_rays(c + _unit(rng, len(idx)) * r * rng.uniform(0, 0.9, (len(idx), 1)).astype(np.float32), _unit(rng, len(idx))))
        src = (c + _unit(rng, len(idx)) * (r * 3.0 + 1.0)).astype(np.float32)
        parts.append(_rays(src, c - src))
        to_c = c - src
        perp = np.cross(to_c, _unit(rng, len(idx)))
        perp /= np.linalg.norm(perp, axis=1, keepdims=True) + 1e-30
        for f in (1.0, 1.0 - 1e-6, 1.0 + 1e-6):
            parts.append(_rays(src, (c + perp * r * f - src).astype(np.float32)))
    if T:
        idx = rng.integers(0, len(T), size=min(n, 4 * len(T)))
        for w in ((1, 0, 0), (0, 1, 0), (0.5, 0.5, 0), (0, 0.5, 0.5), (1 / 3, 1 / 3, 1 / 3)):   # vertices, edges, centroid
            tgt = np.array([np.add(np.add(np.multiply(w[0], T[i].v0.tuple()), np.multiply(w[1], T[i].v1.tuple())),
                                   np.multiply(w[2], T[i].v2.tuple())) for i in idx], np.float32)
            src = (tgt + _unit(rng, len(idx)) * 2.0).astype(np.float32)
            parts.append(_rays(src, tgt - src))
    # directions with zero components, from the camera origin and a random point
    zd = np.array([(0, 0, -1), (1, 0, 0), (0, -1, 0), (0, 1, 1), (1, 0, -1), (-1, -1, 0), (0, 0, 1e-20), (3e-30, 0, -1)],
                  np.float32)
    for org in (np.array(cam.origin.tuple(), np.float32), o[0]):
        parts.append(_rays(np.broadcast_to(org, zd.shape), zd))
    # origins within 2^-63 of the world's origin, where o.o underflows below 2^-126 (the CULL walk hands these rays to
    # the FILTER walk), and the origin itself
    tiny = np.array([(1e-25, 0, 0), (0, -3e-22, 1e-30), (2.0 ** -70, 2.0 ** -70, -2.0 ** -70), (1e-38, 0, 0),
                     (-2.0 ** -64, 0, 0), (0, 0, 0)], np.float32)
    tiny_o = np.repeat(tiny, 4, axis=0)
    parts.append(_rays(tiny_o, _unit(rng, len(tiny_o))))
    if S:
        tgt = np.array([S[i].center.tuple() for i in rng.integers(0, len(S), size=len(tiny_o))], np.float32)
        parts.append(_rays(tiny_o, tgt - tiny_o))
    rays = np.concatenate(parts)
    # t_max in {+inf, -inf, -1, 0.001, a hit's exact t, the next float below and above it}
    base = reference(ob, world, rays)
    hits = rays[base["prim"] >= 0][: 2 * n]
    ts = base["depth"][base["prim"] >= 0][: 2 * n]
    extra = [rays.copy() for _ in range(4)]
    for e, t in zip(extra, (-INF, -1.0, 0.001, INF)):
        e[:, 3] = t
    for f in (lambda t: t, lambda t: np.nextafter(t, F(-INF)), lambda t: np.nextafter(t, F(INF))):
        h = hits.copy()
        h[:, 3] = f(ts)
        extra.append(h)
    return np.concatenate([rays, extra[0][:n], extra[1][:n], extra[2][:n]] + extra[4:] + [invalid_rays()])


def _camera_vector(cam, u, v):
    """The un-normalised camera vector ((llc + u*horizontal) + v*vertical) - origin, in float32 (camera.rs:84-89)."""
    llc, h, vv, o = (np.array(x.tuple(), np.float32) for x in (cam.lower_left_corner, cam.horizontal, cam.vertical,
                                                               cam.origin))
    return ((llc + h * F(u)) + vv * F(v)) - o


def camera_vectors(cam, W, H):
    """The camera vector of every pixel centre (fixed jitter), top row first, float32 [H*W, 3]."""
    cols = np.arange(W, dtype=np.float32)
    rows = (H - 1 - np.arange(H)).astype(np.float32)
    u = (cols + F(0.5)) / F(W - 1)
    v = (rows + F(0.5)) / F(H - 1)
    llc, h, vv, o = (np.array(x.tuple(), np.float32) for x in (cam.lower_left_corner, cam.horizontal, cam.vertical,
                                                               cam.origin))
    U, V = np.meshgrid(u, v)
    p = ((llc[None, None, :] + h[None, None, :] * U[..., None]) + vv[None, None, :] * V[..., None]) - o[None, None, :]
    return p.reshape(-1, 3).astype(np.float32)


# ---------------------------------------------------------------------------------------------------------- C ABI

def test_header_declares_the_call_and_the_package_exports_it(rt, tmp_path):
    text = (ROOT / "include" / "raytracer_b200.h").read_text()
    assert "int rt_trace_rays_device(" in text and "typedef struct RtRay " in text and "typedef struct RtRayQueryOptions" in text
    assert "rt_trace_rays_device" in rt.EXPORTED_SYMBOLS and hasattr(rt.lib(), "rt_trace_rays_device")
    assert rt.lib().rt_abi_version() == 2
    src = tmp_path / "layout.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "raytracer_b200.h"\n'
                   "int main(void) { printf(\"%zu %zu %zu %zu %zu %zu %zu %zu %zu\\n\", sizeof(RtRay), offsetof(RtRay, t_max), "
                   "offsetof(RtRay, direction), offsetof(RtRay, reserved), sizeof(RtRayQueryOptions), "
                   "offsetof(RtRayQueryOptions, flags), offsetof(RtRayQueryOptions, device), "
                   "offsetof(RtRayQueryOptions, reserved), offsetof(RtRayQueryOptions, stats)); return 0; }\n")
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-std=c11", "-I", str(ROOT / "include"), str(src), "-o", str(exe)], check=True)
    got = tuple(map(int, subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()))
    o = rt._RayQueryOptions
    assert got == (32, 12, 16, 28, C.sizeof(o), o.flags.offset, o.device.offset, o.reserved.offset, o.stats.offset)
    assert got[4:] == (24, 4, 8, 12, 16)


def _host_out(n):
    return {"depth": np.full(n, 7.0, np.float32), "position": np.full((n, 3), 7.0, np.float32),
            "normal": np.full((n, 3), 7.0, np.float32), "albedo": np.full((n, 3), 7.0, np.float32),
            "prim": np.full(n, 7, np.int32)}


def _untouched(out):
    return all((b == 7).all() for b in out.values())


def _raw_call(rt, handle, n, rays_addr, out, which=NAMES, options=None, opt_ptr=True, hits=True):
    L = rt.lib()
    o = (options if options is not None else rt.RayQueryOptions())._c(None)
    b = rt.AovBuffers(C.sizeof(rt.AovBuffers), 0, *((out[k].ctypes.data if k in which else None) for k in NAMES))
    rc = L.rt_trace_rays_device(handle.ptr if handle is not None else None, C.byref(o) if opt_ptr else None, n,
                                rays_addr, C.byref(b) if hits else None, None)
    return rc, rt.last_error()


def test_rejections_happen_on_the_host_before_any_device_work(rt, scenes):
    h = rt.load_world(scenes.example_world())
    rays = np.zeros((4 + 1, 8), np.float32)                 # one spare record to misalign by
    base = rays.ctypes.data
    aligned = base if base % 16 == 0 else base + (16 - base % 16)
    assert aligned + 4 * 32 <= base + rays.nbytes
    cases_ = [
        (dict(handle=None), "NULL world handle"),
        (dict(opt_ptr=False), "options is NULL"),
        (dict(options=rt.RayQueryOptions(flags=rt.OPT_FAST_MATH)), "only RT_OPT_GROUP_CULL"),
        (dict(options=rt.RayQueryOptions(flags=rt.OPT_FIXED_JITTER)), "only RT_OPT_GROUP_CULL"),
        (dict(options=rt.RayQueryOptions(flags=0x4)), "only RT_OPT_GROUP_CULL"),
        (dict(hits=False), "hits is NULL"),
        (dict(n=0), "n must be at least 1"),
        (dict(n=2 ** 31), "n must be at most 2^31 - 1"),
        (dict(rays_addr=None), "the ray buffer is NULL"),
        (dict(rays_addr=aligned + 4), "not 16-byte aligned"),
        (dict(rays_addr=aligned + 8), "not 16-byte aligned"),
        (dict(which=()), "every output is NULL"),
    ]
    for kw, text in cases_:
        out = _host_out(4)
        args = dict(handle=h, n=4, rays_addr=aligned, out=out)
        args.update(kw)
        rc, err = _raw_call(rt, **args)
        assert rc != 0 and text in err, (kw, err)
        assert _untouched(out)


def test_wrong_struct_size_is_rejected(rt, scenes):
    h = rt.load_world(scenes.example_world())
    out = _host_out(2)
    rays = np.zeros((2, 8), np.float32)
    b = rt.AovBuffers(C.sizeof(rt.AovBuffers), 0, *(out[k].ctypes.data for k in NAMES))
    for size in (0, 16, 32):
        o = rt._RayQueryOptions(size, 0, -1, 0, None)
        assert rt.lib().rt_trace_rays_device(h.ptr, C.byref(o), 2, rays.ctypes.data, C.byref(b), None) != 0
        assert "struct_size must be sizeof(RtRayQueryOptions)" in rt.last_error()
        assert _untouched(out)


def test_overlapping_outputs_are_rejected(rt, scenes):
    h = rt.load_world(scenes.example_world())
    n = 8
    blob = np.full(4096, 7, np.uint8)
    base = blob.ctypes.data + (-blob.ctypes.data) % 16
    rays = base                                               # [0, 256)
    layout = {"depth": 1024, "position": 1536, "normal": 2048, "albedo": 2560, "prim": 3072}
    L = rt.lib()
    o = rt.RayQueryOptions()._c(None)

    def call(**moved):
        addr = {k: base + v for k, v in layout.items()}
        addr.update({k: base + v for k, v in moved.items()})
        b = rt.AovBuffers(C.sizeof(rt.AovBuffers), 0, *(addr[k] for k in NAMES))
        assert L.rt_trace_rays_device(h.ptr, C.byref(o), n, rays, C.byref(b), None) != 0
        return rt.last_error()

    assert "the depth output overlaps the rays" in call(depth=255)
    assert "the prim output overlaps the rays" in call(prim=0)
    assert "the normal output overlaps the position output" in call(normal=1536 + 95)
    assert "the prim output overlaps the albedo output" in call(prim=2560 + 64)
    assert (blob == 7).all()
    # adjacent ranges do not overlap: the call gets as far as the device (none here, or host memory)
    err = call(depth=256)
    assert "overlaps" not in err


def test_valid_call_never_falls_back(rt, scenes):
    """A valid call with host arrays fails — without a device because there is none, with one because the arrays are
    not device memory — and never writes an output on the CPU."""
    h = rt.load_world(scenes.example_world())
    rays = _rays([0.0, 0.0, 0.0], [0.0, 0.0, -1.0])
    assert rays.ctypes.data % 16 == 0
    out = _host_out(1)
    rc, err = _raw_call(rt, h, 1, rays.ctypes.data, out, options=rt.RayQueryOptions(group_cull=True))
    want = "no CUDA device available" if rt.device_count() == 0 else "buffer is not device memory of device"
    assert rc != 0 and want in err, err
    assert _untouched(out)


# --------------------------------------------------------------------------------------------------- references

def test_known_answers_on_world_txt(ob, scenes):
    """world.txt: a ray from the origin along (0,0,-1) hits the sphere `0 0 -1 r 0.5` at t = 0.5 with normal (0,0,1);
    with t_max = 0.5 it misses (strict sphere window), with nextafter(0.5, inf) it hits."""
    cam, world = ob.parse_input(scenes.default_world())
    idx = [i for i, s in enumerate(world.spheres()) if s.center.tuple() == (0.0, 0.0, -1.0) and s.radius == 0.5]
    assert len(idx) == 1
    rays = np.concatenate([_rays([0.0, 0.0, 0.0], [0.0, 0.0, -1.0], t) for t in (INF, 0.5, np.nextafter(F(0.5), F(INF)))]
                          + [_rays([0.0, 0.0, 0.0], [0.0, 0.0, -7.0])])
    out = reference(ob, world, rays)
    for i in (0, 2, 3):
        assert out["prim"][i] == idx[0] and out["depth"][i] == F(0.5)
        assert tuple(out["position"][i]) == (0.0, 0.0, -0.5) and tuple(out["normal"][i]) == (0.0, 0.0, 1.0)
    assert out["prim"][1] == -1 and np.isinf(out["depth"][1]) and (out["position"][1] == 0).all()
    assert out["albedo"][1][2] == 1.0                                   # the sky colour of the ray
    assert_same(out, literal_records(world, rays))


def test_triangle_hit_at_exactly_t_max_is_kept(ob):
    world = ob.World()
    world.add_triangle((-1.0, -1.0, -2.0), (1.0, -1.0, -2.0), (0.0, 1.0, -2.0), ob.material(ob.DIFFUSE, (0.2, 0.4, 0.6)))
    rays = _rays([0.0, 0.0, 0.0], [0.0, 0.0, -1.0])
    t = reference(ob, world, rays)["depth"][0]
    assert t == F(2.0)
    rays = np.concatenate([_rays([0.0, 0.0, 0.0], [0.0, 0.0, -1.0], x) for x in (t, np.nextafter(t, F(-INF)))])
    out = reference(ob, world, rays)
    assert out["prim"].tolist() == [0, -1]
    assert out["albedo"][0].tolist() == [F(0.2), F(0.4), F(0.6)]
    assert_same(out, literal_records(world, rays))


def test_invalid_rays_give_the_invalid_record(ob, scenes):
    cam, world = ob.parse_input(scenes.default_world())
    rays = invalid_rays()
    out = reference(ob, world, rays)
    bad = out["prim"] == -2
    assert bad.sum() >= 20 and (~bad).sum() >= 8
    assert (out["depth"][bad].view(np.uint32) == 0x7FFFFFFF).all()
    for k in ("position", "normal", "albedo"):
        assert (out[k][bad].view(np.uint32) == 0).all()
    assert_same(out, literal_records(world, rays))


@pytest.mark.parametrize("case", cases.SMALL_CASES, ids=[c[0] for c in cases.SMALL_CASES])
def test_reference_equals_literal_restatement_on_small_cases(ob, scenes, case):
    name, key, camera, W, H, spp, depth, fixed = case
    cam, world = cases.oracle_scene(ob, scenes, key, camera)
    n = 24 if world.n_spheres + world.n_triangles < 100 else 6
    rays = families(ob, world, cam, seed=zlib.crc32(name.encode()) & 0xFFFF, n=n)
    if world.n_spheres + world.n_triangles >= 100:
        rays = rays[np.random.default_rng(1).permutation(len(rays))[:160]]
    assert_same(reference(ob, world, rays), literal_records(world, rays))


@pytest.mark.parametrize("seed", range(20))
def test_reference_equals_literal_restatement_on_random_worlds(ob, seed):
    cam, world = ob.parse_input(cases.random_world(seed, n_spheres=12, n_triangles=10))
    rays = families(ob, world, cam, seed=seed, n=12)
    assert_same(reference(ob, world, rays), literal_records(world, rays))


# ---------------------------------------------------------------------------------------- device function on the host

def _load_hostsim(name):
    subprocess.run(["make", "-C", str(RAYS_HOST), "build/" + name], check=True, capture_output=True)
    L = C.CDLL(str(RAYS_HOST / "build" / name))
    L.hostsim_trace_rays.restype = C.c_int
    L.hostsim_trace_rays.argtypes = [C.c_char_p, C.c_size_t, C.c_void_p, C.c_uint32] + [C.c_void_p] * 5
    return L


@pytest.fixture(scope="module")
def hostsim():
    return _load_hostsim("librays_hostsim.so")


@pytest.fixture(scope="module")
def hostsim_perturbed():
    return _load_hostsim("librays_hostsim_perturb.so")


def _hostsim(L, text, rays, walk):
    rays = np.ascontiguousarray(rays, np.float32)
    out = _empty(len(rays))
    rc = L.hostsim_trace_rays(text.encode(), len(rays), rays.ctypes.data, walk, *(out[k].ctypes.data for k in NAMES))
    assert rc == 0, rc
    return out


def _walks(world):
    return (0, 0x80000000) + ((0x40000000,) if world.n_spheres >= 64 else ())


@pytest.mark.parametrize("case", cases.SMALL_CASES, ids=[c[0] for c in cases.SMALL_CASES])
def test_device_function_on_host_equals_reference(hostsim, ob, scenes, case):
    name, key, camera, W, H, spp, depth, fixed = case
    cam, world = cases.oracle_scene(ob, scenes, key, camera)
    text = cases.scene_text(scenes, key)
    rays = families(ob, world, cam, seed=7 + (zlib.crc32(name.encode()) & 0xFFFF), n=96)
    want = reference(ob, world, rays)
    for walk in _walks(world):
        assert_same(_hostsim(hostsim, text, rays, walk), want)


@pytest.mark.parametrize("seed", range(50))
def test_device_function_on_random_worlds(hostsim, ob, seed):
    text = cases.random_world(seed)
    cam, world = ob.parse_input(text)
    rays = families(ob, world, cam, seed=1000 + seed, n=48)
    want = reference(ob, world, rays)
    for walk in (0, 0x80000000, 0x40000000):
        assert_same(_hostsim(hostsim, text, rays, walk), want)


@pytest.mark.parametrize("seed", range(40, 50))
def test_device_function_with_perturbed_reciprocals(hostsim_perturbed, ob, seed):
    text = cases.random_world(seed, n_spheres=66, n_triangles=40)
    cam, world = ob.parse_input(text)
    rays = families(ob, world, cam, seed=seed, n=48)
    want = reference(ob, world, rays)
    for walk in (0, 0x80000000, 0x40000000):
        assert_same(_hostsim(hostsim_perturbed, text, rays, walk), want)


def test_device_function_on_invalid_rays(hostsim, ob, scenes):
    for text in (scenes.default_world(), cases.random_world(3)):
        cam, world = ob.parse_input(text)
        rays = invalid_rays()
        want = reference(ob, world, rays)
        for walk in _walks(world):
            assert_same(_hostsim(hostsim, text, rays, walk), want)


def test_camera_vectors_give_the_first_hit_record_on_host(hostsim, ob, scenes):
    """The un-normalised camera vector of a pixel centre is the camera ray: same record as the first-hit buffers."""
    import test_aov
    cam, world = ob.parse_input(scenes.example_world())
    W, H = 40, 24
    want = test_aov.primary_hits(ob, world, cam, W, H, fixed_jitter=True)
    rays = _rays(np.array(cam.origin.tuple(), np.float32), camera_vectors(cam, W, H))
    got = _hostsim(hostsim, scenes.example_world(), rays, 0)
    assert_same({k: v.reshape(want[k].shape) for k, v in got.items()}, want)


# ------------------------------------------------------------------------------------------------------------ GPU

def _gpu(gpu_rt, handle, rays, cull=False, stats=None, outputs=NAMES):
    import torch
    r = torch.from_numpy(np.ascontiguousarray(rays, np.float32)).cuda()
    out = {k: torch.full(s, 7, dtype=dt, device="cuda") for k, (s, dt) in
           {"depth": ((len(rays),), torch.float32), "position": ((len(rays), 3), torch.float32),
            "normal": ((len(rays), 3), torch.float32), "albedo": ((len(rays), 3), torch.float32),
            "prim": ((len(rays),), torch.int32)}.items()}
    torch.cuda.synchronize()
    gpu_rt.trace_rays_device(handle, gpu_rt.RayQueryOptions(group_cull=cull), len(rays), r.data_ptr(),
                             **{k: (out[k].data_ptr() if k in outputs else 0) for k in NAMES}, stats=stats)
    return {k: v.cpu().numpy() for k, v in out.items()}


@pytest.mark.gpu
@pytest.mark.parametrize("case", cases.SMALL_CASES, ids=[c[0] for c in cases.SMALL_CASES])
def test_gpu_small_cases(gpu_rt, ob, scenes, case):
    name, key, camera, W, H, spp, depth, fixed = case
    cam, world = cases.oracle_scene(ob, scenes, key, camera)
    h = cases.product_scene(gpu_rt, scenes, key, camera)
    rays = families(ob, world, cam, seed=11 + (zlib.crc32(name.encode()) & 0xFFFF), n=256)
    want = reference(ob, world, rays)
    for cull in ((False, True) if world.n_spheres >= 64 else (False,)):
        st = gpu_rt.RenderStats()
        assert_same(_gpu(gpu_rt, h, rays, cull, st), want, canonical_nan=True)
        assert st.rays == len(rays) and st.samples == len(rays) and st.launches == 1 and st.culled == int(cull)


@pytest.mark.gpu
def test_gpu_camera_vectors_equal_render_aov(gpu_rt, ob, scenes):
    """For every small case's camera: the camera vectors of the pixel centres, through the ray query, give
    render_aov's buffers (fixed jitter) bit for bit."""
    for name, key, camera, W, H, spp, depth, fixed in cases.SMALL_CASES:
        cam, world = cases.oracle_scene(ob, scenes, key, camera)
        h = cases.product_scene(gpu_rt, scenes, key, camera)
        aov = {k: v.cpu().numpy() for k, v in gpu_rt.render_aov(h, W, H, gpu_rt.Options(fixed_jitter=True)).items()}
        rays = _rays(np.array(cam.origin.tuple(), np.float32), camera_vectors(cam, W, H))
        got = _gpu(gpu_rt, h, rays)
        assert_same({k: v.reshape(aov[k].shape) for k, v in got.items()}, aov)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 31, 33, 1000, 2 ** 20 + 7])
def test_gpu_sizes(gpu_rt, ob, scenes, n):
    cam, world = ob.parse_input(scenes.example_world())
    h = gpu_rt.load_world(scenes.example_world())
    base = families(ob, world, cam, seed=n % 1000, n=64)
    rays = base[np.random.default_rng(n).integers(0, len(base), size=n)]
    assert_same(_gpu(gpu_rt, h, rays), reference(ob, world, rays), canonical_nan=True)


@pytest.mark.gpu
def test_gpu_empty_world_and_four_materials(gpu_rt, ob):
    import test_aov
    h = gpu_rt.world_new((0.0, 0.0, 0.0), 1.5)
    rays = np.concatenate([_rays([0.0, 0.0, 0.0], _unit(np.random.default_rng(3), 500)), invalid_rays()])
    got = _gpu(gpu_rt, h, rays)
    assert set(np.unique(got["prim"])) == {-1, -2}
    assert_same(got, reference(ob, ob.World(), rays), canonical_nan=True)
    h, world, cam = test_aov._four_material_worlds(gpu_rt, ob)
    rays = families(ob, world, cam, seed=5, n=400)
    got = _gpu(gpu_rt, h, rays)
    assert set(np.unique(got["prim"])) >= {-2, -1, 0, 1, 2, 3, 5}
    assert_same(got, reference(ob, world, rays), canonical_nan=True)


@pytest.mark.gpu
def test_gpu_global_memory_path_filter_and_cull(gpu_rt, ob, scenes):
    text = scenes.synthetic_world(16000, 0, seed=4242)            # hot lists larger than shared memory
    cam, world = ob.parse_input(text)
    h = gpu_rt.load_world(text)
    rays = families(ob, world, cam, seed=9, n=128)
    # origins so close to the world's origin that o.o underflows (the CULL walk's fallback)
    tiny = _rays([[1e-25, 0.0, 0.0], [0.0, -3e-22, 1e-30], [0.0, 0.0, 0.0]], _unit(np.random.default_rng(4), 3))
    rays = np.concatenate([rays, tiny, _rays(tiny[:, 0:3], camera_vectors(cam, 4, 2)[:3])])
    want = reference(ob, world, rays)
    for cull in (False, True):
        st = gpu_rt.RenderStats()
        assert_same(_gpu(gpu_rt, h, rays, cull, st), want, canonical_nan=True)
        assert st.resident == 0 and st.smem_bytes == 0 and st.filtered == 1 and st.culled == int(cull)


@pytest.mark.gpu
@pytest.mark.parametrize("key,n", [("c3", 2 ** 18), ("c5", 2 ** 14)])
def test_gpu_large_worlds(gpu_rt, ob, scenes, key, n):
    cam, world = cases.oracle_scene(ob, scenes, key, "file")
    h = cases.product_scene(gpu_rt, scenes, key, "file")
    rng = np.random.default_rng(n)
    lo, hi = _bounds(world)
    o = (lo + rng.uniform(size=(n, 3)) * (hi - lo)).astype(np.float32)
    o[: n // 2] = np.array(cam.origin.tuple(), np.float32)
    rays = _rays(o, _unit(rng, n) * np.exp2(rng.integers(-20, 21, size=(n, 1))).astype(np.float32))
    rays[::7, 3] = rng.uniform(0.0, 5.0, size=len(rays[::7]))
    want = reference(ob, world, rays)
    for cull in (False, True):
        st = gpu_rt.RenderStats()
        assert_same(_gpu(gpu_rt, h, rays, cull, st), want, canonical_nan=True)
        assert st.filtered == 1 and st.resident == 1 and st.culled == int(cull)


@pytest.mark.gpu
def test_gpu_each_output_alone(gpu_rt, ob, scenes):
    cam, world = ob.parse_input(scenes.example_world())
    h = gpu_rt.load_world(scenes.example_world())
    rays = families(ob, world, cam, seed=21, n=64)
    want = reference(ob, world, rays)
    for k in NAMES:
        got = _gpu(gpu_rt, h, rays, outputs=(k,))
        assert_same(got, want, canonical_nan=True, keys=(k,))
        assert all((got[j] == 7).all() for j in NAMES if j != k)


@pytest.mark.gpu
def test_gpu_caller_stream_and_explicit_device(gpu_rt, ob, scenes):
    import torch
    torch.cuda.set_device(0)
    cam, world = ob.parse_input(scenes.c3_world())
    h = gpu_rt.load_world(scenes.c3_world())
    rays = families(ob, world, cam, seed=31, n=512)
    want = reference(ob, world, rays)
    s = torch.cuda.Stream()
    r = torch.from_numpy(rays).cuda()
    out = {"depth": torch.full((len(rays),), 7.0, device="cuda"), "position": torch.full((len(rays), 3), 7.0, device="cuda"),
           "normal": torch.full((len(rays), 3), 7.0, device="cuda"), "albedo": torch.full((len(rays), 3), 7.0, device="cuda"),
           "prim": torch.full((len(rays),), 7, dtype=torch.int32, device="cuda")}
    torch.cuda.synchronize()
    with torch.cuda.stream(s):
        torch.cuda._sleep(200_000_000)                              # ~0.1 s of work ahead of the kernel on the stream
    gpu_rt.trace_rays_device(h, gpu_rt.RayQueryOptions(device=0), len(rays), r.data_ptr(),
                             *(out[k].data_ptr() for k in NAMES), stream=s.cuda_stream)
    assert not s.query(), "the call waited for the caller's stream"
    assert torch.cuda.current_device() == 0
    s.synchronize()
    assert_same({k: v.cpu().numpy() for k, v in out.items()}, want, canonical_nan=True)


@pytest.mark.gpu
def test_gpu_trace_rays_waits_for_torch_default_stream(gpu_rt, ob, scenes):
    """trace_rays with stream=None packs the rays on torch's current stream — here the legacy default stream, behind
    ~0.1 s of work — and its kernel must run after that packing, not on a stream that does not wait for it."""
    import torch
    torch.cuda.set_device(0)
    assert torch.cuda.current_stream().cuda_stream == 0
    cam, world = ob.parse_input(scenes.c3_world())
    h = gpu_rt.load_world(scenes.c3_world())
    rays = families(ob, world, cam, seed=51, n=2048)
    rays[:, 7] = 0.0
    want = reference(ob, world, rays)
    o = torch.from_numpy(rays[:, 0:3].copy()).cuda()
    d = torch.from_numpy(rays[:, 4:7].copy()).cuda()
    t = torch.from_numpy(rays[:, 3].copy()).cuda()
    junk = torch.full((len(rays), 8), float("nan"), device="cuda")   # the block the packed rays will likely reuse
    del junk
    torch.cuda.synchronize()
    torch.cuda._sleep(200_000_000)                                  # ahead of the packing on torch's stream
    got = {k: v.cpu().numpy() for k, v in gpu_rt.trace_rays(h, o, d, t).items()}
    assert_same(got, want, canonical_nan=True)


@pytest.mark.gpu
def test_gpu_stats(gpu_rt, scenes):
    import torch
    h = gpu_rt.load_world(scenes.c3_world())
    n = 100_000
    st = gpu_rt.RenderStats()
    o = torch.zeros((n, 3), device="cuda")
    d = torch.randn((n, 3), device="cuda")
    gpu_rt.trace_rays(h, o, d, stats=st)
    assert st.rays == n and st.samples == n and st.launches == 1
    assert st.kernel_ms > 0 and st.total_ms >= st.kernel_ms and st.grid >= 1 and st.block in (256, 1024)
    assert st.resident == 1 and st.smem_bytes > 0 and st.filtered == 1 and st.culled == 0


@pytest.mark.gpu
def test_gpu_trace_rays_tensors(gpu_rt, ob, scenes):
    import torch
    cam, world = ob.parse_input(scenes.default_world())
    h = gpu_rt.load_world(scenes.default_world())
    rays = families(ob, world, cam, seed=41, n=128)
    rays[:, 7] = 0.0                                              # trace_rays packs reserved = 0
    o = torch.from_numpy(rays[:, 0:3].copy()).cuda()
    d = torch.from_numpy(rays[:, 4:7].copy()).cuda()
    t = torch.from_numpy(rays[:, 3].copy()).cuda()
    got = {k: v.cpu().numpy() for k, v in gpu_rt.trace_rays(h, o, d, t).items()}
    assert_same(got, reference(ob, world, rays), canonical_nan=True)
    for t_max in (None, 0.75):
        r = rays.copy()
        r[:, 3] = INF if t_max is None else t_max
        got = {k: v.cpu().numpy() for k, v in gpu_rt.trace_rays(h, o, d, t_max).items()}
        assert_same(got, reference(ob, world, r), canonical_nan=True)
    got = gpu_rt.trace_rays(h, o, d, outputs=("prim",), cull=False, device=0)
    assert set(got) == {"prim"}
    empty = gpu_rt.trace_rays(h, o[:0], d[:0])
    assert {k: tuple(v.shape) for k, v in empty.items()} == {"depth": (0,), "position": (0, 3), "normal": (0, 3),
                                                              "albedo": (0, 3), "prim": (0,)}
    s = torch.cuda.Stream()
    got = gpu_rt.trace_rays(h, o, d, stream=s)
    s.synchronize()
    assert_same({k: v.cpu().numpy() for k, v in got.items()}, reference(ob, world, _rays(rays[:, 0:3], rays[:, 4:7])),
                canonical_nan=True)
