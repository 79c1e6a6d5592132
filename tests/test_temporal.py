"""Temporal accumulation (rt_temporal_accumulate_device / temporal_accumulate / TemporalRenderer): a frame's colour sums
blended with the previous frame's colour history, reprojected through the first-hit buffers, equal to the numpy
reference below bit for bit.

`temporal_reference` restates DESIGN.md §15.1 in numpy float32, vectorised over pixels, with the four bilinear taps in
the kernel's order.  A skipped tap adds +0.0 to the sums, which leaves them unchanged (they start at +0.0 and so are
never -0.0), so the masked sums equal the kernel's branchy ones.

CPU tests: the boundary (symbols, struct layout, defaults, every rejection), the device header's per-pixel functions
built for the host (tests/temporal_host) against the reference on random and oracle frames, known answers (first frame,
static camera, disocclusion traced with the ray reference) and the quality along a camera path.  GPU tests: the kernel
against the reference on frames the library renders.  Between the GPU and the CPU a NaN is compared as "NaN".
"""
import ctypes as C
import re
import subprocess
from pathlib import Path

import numpy as np
import pytest

import cases

HERE = Path(__file__).resolve().parent
ROOT = HERE.parent
TEMPORAL_HOST = HERE / "temporal_host"
f32 = np.float32
MIN_WEIGHT = f32(2.0 ** -7)                                                  # §15.1: accepted weight below: no history
DEFAULTS = {"max_history": 8, "normal_cos": 0.9, "plane_tol": 0.02}
PATH_STEP = (0.04, 0.0, 0.02)                                                # camera move per frame (move_camera_position)


# ------------------------------------------------------------------------------------------------------- reference

def _dot(a, b):
    """§15.1: (a.x*b.x + a.y*b.y) + a.z*b.z"""
    return (a[..., 0] * b[..., 0] + a[..., 1] * b[..., 1]) + a[..., 2] * b[..., 2]


def _cross(a, b):
    """§15.1: (a.y*b.z - a.z*b.y, a.z*b.x - a.x*b.z, a.x*b.y - a.y*b.x)"""
    return np.array([a[1] * b[2] - a[2] * b[1], a[2] * b[0] - a[0] * b[2], a[0] * b[1] - a[1] * b[0]], np.float32)


def project(prev_camera, X, W, H):
    """The continuous previous pixel (x, y) of the points X [..., 3] and whether it counts (in front of the previous
    camera, not NaN, inside [-1, W] x [-1, H])."""
    c = np.asarray(prev_camera, np.float32)
    o, L, h, v = c[0:3], c[3:6], c[6:9], c[9:12]
    a = (L - o).astype(np.float32)
    cn, cs, ct = _cross(h, v), _cross(v, a), _cross(a, h)
    det = _dot(a, cn)
    with np.errstate(all="ignore"):
        w = (X - o).astype(np.float32)
        den = _dot(w, cn)
        front = (den != 0) & ((den > 0) == (det > 0))
        u = _dot(w, cs) / den
        t = _dot(w, ct) / den
        x = u * f32(W - 1) - f32(0.5)
        r = t * f32(H - 1) - f32(0.5)
        y = f32(H - 1) - r
        ok = front & (x >= -1) & (x <= f32(W)) & (y >= -1) & (y <= f32(H))
    return x, y, ok


def _f32_as_u8(x):
    """Rust `f32 as u8`: truncate, saturate, NaN -> 0."""
    with np.errstate(invalid="ignore"):
        t = np.where(x > 0, np.minimum(np.trunc(np.nan_to_num(x, nan=0.0)), 255), 0)
    return t.astype(np.uint8)


def rgba8(c):
    """resolve_pixel<false>(r, g, b, a, 1) (rt_trace.cuh): sqrt gamma, x255.999, `as u8`; k = 1.0f / 1."""
    one, q = f32(1), f32(255.999)
    with np.errstate(invalid="ignore"):
        rgb = [_f32_as_u8(np.sqrt(c[..., i] * one) * q) for i in range(3)]
    return np.stack(rgb + [_f32_as_u8((c[..., 3] * one) * q)], axis=-1)


def temporal_reference(accum, spp, position, normal, prim, camera, prev=None, max_history=0, normal_cos=0.0,
                       plane_tol=0.0):
    """{"color": float32 [H,W,4], "length": float32 [H,W], "pixels": uint8 [H,W,4]} of DESIGN.md §15.1.  prev: None or
    {"camera", "position", "normal", "prim", "color", "length"} of the previous frame; a 0 option takes its default."""
    accum, position, normal = (np.asarray(a, np.float32) for a in (accum, position, normal))
    prim = np.asarray(prim)
    H, W = prim.shape
    mh = f32(max_history or DEFAULTS["max_history"])
    nc = f32(normal_cos or DEFAULTS["normal_cos"])
    pt = f32(plane_tol or DEFAULTS["plane_tol"])
    with np.errstate(all="ignore"):
        color = accum * (f32(1) / f32(spp))                                  # the mean, alpha included
        length = np.full((H, W), f32(spp), np.float32)
        if prev is not None:
            cam, pcam = np.asarray(camera, np.float32), np.asarray(prev["camera"], np.float32)
            pprim, pnormal, pposition = (np.asarray(prev[k]) for k in ("prim", "normal", "position"))
            pcolor, plength = np.asarray(prev["color"], np.float32), np.asarray(prev["length"], np.float32)
            hit = (prim >= 0) & np.isfinite(position).all(-1) & np.isfinite(normal).all(-1)
            rows, cols = np.mgrid[0:H, 0:W]
            if cam.tobytes() == pcam.tobytes():                              # identity rule
                taps = [(cols, rows, np.ones((H, W), np.float32), hit)]
            else:
                x, y, ok = project(pcam, position, W, H)
                ok = ok & hit
                x0, y0 = np.floor(x), np.floor(y)
                fx, fy = x - x0, y - y0
                ix = np.where(ok, x0, 0).astype(np.int64)
                iy = np.where(ok, y0, 0).astype(np.int64)
                one = f32(1)
                taps = [(ix, iy, (one - fx) * (one - fy), ok), (ix + 1, iy, fx * (one - fy), ok),
                        (ix, iy + 1, (one - fx) * fy, ok), (ix + 1, iy + 1, fx * fy, ok)]
            sw = np.zeros((H, W), np.float32)
            sc = np.zeros((H, W, 4), np.float32)
            sl = np.zeros((H, W), np.float32)
            for qx, qy, wt, ok in taps:                                      # tap order
                inside = ok & (qx >= 0) & (qy >= 0) & (qx < W) & (qy < H) & (wt > 0)
                cx, cy = np.clip(qx, 0, W - 1), np.clip(qy, 0, H - 1)
                acc = inside & (pprim[cy, cx] >= 0)
                acc &= _dot(normal, pnormal[cy, cx]) >= nc
                acc &= np.abs(_dot(normal, pposition[cy, cx] - position)) <= pt
                sw = sw + np.where(acc, wt, f32(0))
                sc = sc + np.where(acc[..., None], wt[..., None] * pcolor[cy, cx], f32(0))
                sl = sl + np.where(acc, wt * plength[cy, cx], f32(0))
            n = np.fmin(sl / sw, mh)                                         # fminf: a NaN length gives max_history
            use = (sw >= MIN_WEIGHT) & (n > 0)
            L = n + f32(spp)
            blended = ((sc / sw[..., None]) * n[..., None] + accum) / L[..., None]
            color = np.where(use[..., None], blended, color)
            length = np.where(use, L, length)
    return {"color": color, "length": length, "pixels": rgba8(color)}


def _bits(a, canonical_nan=False):
    a = np.ascontiguousarray(a)
    if a.dtype != np.float32:
        return a
    b = a.view(np.uint32).copy()
    if canonical_nan:
        b[np.isnan(a)] = 0x7FFFFFFF
    return b


def assert_same(got, want, canonical_nan=False):
    for k in ("color", "length", "pixels"):
        if got.get(k) is None:
            continue
        g, w = np.asarray(got[k]), np.asarray(want[k])
        bad = np.argwhere(_bits(g, canonical_nan) != _bits(w, canonical_nan))
        assert bad.size == 0, f"{k}: {len(bad)} values differ, first at {bad[0].tolist()}: {g[tuple(bad[0])]} vs {w[tuple(bad[0])]}"


# ----------------------------------------------------------------------------------------------- random frames

def _camera(origin, aspect=1.5, yaw=0.0):
    """12 floats of a pinhole camera looking down -z (rotated by `yaw` about y), viewport 2*aspect x 2 at distance 1."""
    o = np.float32(origin)
    cy, sy = np.cos(yaw), np.sin(yaw)
    right, up, fwd = np.float32([cy, 0, -sy]), np.float32([0, 1, 0]), np.float32([-sy, 0, -cy])
    h, v = right * f32(2 * aspect), up * f32(2)
    L = o + fwd - h / 2 - v / 2
    return np.concatenate([o, L, h, v]).astype(np.float32)


def _point(camera, u, t, s):
    """o + s * ((L + h u) + v t - o): the point at parameter s on the camera ray of (u, t)."""
    c = np.asarray(camera, np.float32)
    d = (c[3:6] + c[6:9] * np.float32(u)[..., None]) + c[9:12] * np.float32(t)[..., None] - c[0:3]
    return (c[0:3] + np.float32(s)[..., None] * d).astype(np.float32)


def random_frames(seed, W, H, nasty=True):
    """(current inputs, prev dict) of a random scene seen from two nearby cameras: positions on the current camera's
    rays, previous guides near them, and, with `nasty`: misses, NaN / inf guides, zero, fractional and NaN lengths,
    points behind the previous camera, and points that project onto the previous frame's border and just past it."""
    rng = np.random.default_rng(seed)
    cam = _camera((0.0, 0.0, 0.0))
    pcam = _camera((rng.uniform(-0.1, 0.1), rng.uniform(-0.05, 0.05), rng.uniform(-0.1, 0.1)), yaw=rng.uniform(-0.05, 0.05))
    u = (np.arange(W, dtype=np.float32)[None, :] + f32(0.5)) / f32(max(W - 1, 1)) * np.ones((H, 1), np.float32)
    t = (np.float32(H - 1) - np.arange(H, dtype=np.float32)[:, None] + f32(0.5)) / f32(max(H - 1, 1)) * np.ones((1, W), np.float32)
    s = rng.uniform(2, 6, (H, W)).astype(np.float32)
    position = _point(cam, u, t, s)
    normal = rng.normal(size=(H, W, 3)).astype(np.float32)
    normal /= np.linalg.norm(normal, axis=-1, keepdims=True).astype(np.float32)
    normal[rng.random((H, W)) < 0.6] = np.float32([0, 0, 1])                # large flat regions
    prim = rng.integers(0, 5, (H, W)).astype(np.int32)
    accum = (rng.random((H, W, 4)) * 8).astype(np.float32)
    accum[..., 3] = 3.0
    # the previous frame: its own pixels' points, jittered off the surface a little, mostly the same normals
    px, py, _ = project(cam, _point(pcam, u, t, s), W, H)
    pposition = _point(pcam, u, t, s) + rng.normal(scale=0.01, size=(H, W, 3)).astype(np.float32)
    pnormal = normal.copy()
    flip = rng.random((H, W)) < 0.2
    pnormal[flip] = np.float32([1, 0, 0])
    pprim = prim.copy()
    pcolor = rng.random((H, W, 4)).astype(np.float32)
    pcolor[..., 3] = 1.0
    plength = rng.integers(1, 40, (H, W)).astype(np.float32)
    if nasty:
        prim[rng.random((H, W)) < 0.1] = -1
        pprim[rng.random((H, W)) < 0.1] = -1
        position[rng.random((H, W)) < 0.02, 1] = np.nan
        normal[rng.random((H, W)) < 0.02, 2] = np.inf
        pnormal[rng.random((H, W)) < 0.02, 0] = np.nan
        plength[rng.random((H, W)) < 0.05] = 0.0
        plength[rng.random((H, W)) < 0.05] *= f32(0.37)
        plength[rng.random((H, W)) < 0.02] = np.nan
        pcolor[rng.random((H, W)) < 0.01, 1] = np.nan
        behind = rng.random((H, W)) < 0.05                                  # behind the previous camera
        position[behind] = pcam[0:3] - (position[behind] - pcam[0:3])
        # points on the previous camera's rays to the border values x = -1, W and y = -1, H, swept over small steps
        k = rng.random((H, W)) < 0.15
        n = int(k.sum())
        if n:
            side = rng.integers(0, 4, n)
            step = (rng.integers(-40, 41, n) * 1e-8).astype(np.float32)
            wm1, hm1 = f32(max(W - 1, 1)), f32(max(H - 1, 1))
            ub = np.where(side == 0, f32(-0.5) / wm1, np.where(side == 1, (f32(W) + f32(0.5)) / wm1, rng.random(n)))
            tb = np.where(side == 2, (f32(H) + f32(0.5)) / hm1, np.where(side == 3, f32(-0.5) / hm1, rng.random(n)))
            ub = (ub + np.where(side < 2, step, 0)).astype(np.float32)
            tb = (tb + np.where(side >= 2, step, 0)).astype(np.float32)
            position[k] = _point(pcam, ub, tb, rng.uniform(2, 6, n))
    prev = {"camera": pcam, "position": pposition, "normal": pnormal, "prim": pprim, "color": pcolor, "length": plength}
    return (accum, position, normal, prim, cam), prev


# ---------------------------------------------------------------------------------------------------------- C ABI

def test_header_declares_the_call_and_the_package_exports_it(rt, tmp_path):
    text = (ROOT / "include" / "raytracer_b200.h").read_text()
    assert "int rt_temporal_accumulate_device(" in text and "typedef struct RtTemporalOptions" in text
    assert "typedef struct RtTemporalHistory" in text
    assert "rt_temporal_accumulate_device" in rt.EXPORTED_SYMBOLS and hasattr(rt.lib(), "rt_temporal_accumulate_device")
    assert rt.lib().rt_abi_version() == 2
    src = tmp_path / "layout.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "raytracer_b200.h"\n'
                   "int main(void) { printf(\"%zu %zu %zu %zu %zu %zu %zu %zu %zu\\n\", sizeof(RtTemporalOptions), "
                   "offsetof(RtTemporalOptions, normal_cos), offsetof(RtTemporalOptions, plane_tol), "
                   "offsetof(RtTemporalOptions, device), offsetof(RtTemporalOptions, stats), sizeof(RtTemporalHistory), "
                   "offsetof(RtTemporalHistory, guides), offsetof(RtTemporalHistory, color), "
                   "offsetof(RtTemporalHistory, length)); return 0; }\n")
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-std=c11", "-I", str(ROOT / "include"), str(src), "-o", str(exe)], check=True)
    got = list(map(int, subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()))
    o, h = rt._TemporalOptions, rt._TemporalHistory
    assert got == [C.sizeof(o), o.normal_cos.offset, o.plane_tol.offset, o.device.offset, o.stats.offset, C.sizeof(h),
                   h.guides.offset, h.color.offset, h.length.offset]


def test_defaults_agree_everywhere(rt):
    """The header's RT_TEMPORAL_DEFAULT_*, the host layer's constants, the package's and this reference's."""
    hdr = (ROOT / "include" / "raytracer_b200.h").read_text()
    host = (ROOT / "rust-swift-raytracer_b200" / "csrc" / "rt_host.hpp").read_text()
    for key, name, cname in (("max_history", "MAX_HISTORY", "MaxHistory"), ("normal_cos", "NORMAL_COS", "NormalCos"),
                             ("plane_tol", "PLANE_TOL", "PlaneTol")):
        h = re.search(r"#define RT_TEMPORAL_DEFAULT_%s ([0-9.]+)[uf]" % name, hdr).group(1)
        c = re.search(r"kTemporalDefault%s\s*=\s*([0-9.]+)[uf];" % cname, host).group(1)
        assert f32(h) == f32(c) == f32(getattr(rt, "TEMPORAL_DEFAULT_" + name)) == f32(DEFAULTS[key]), key


def _host_frame(W=8, H=4):
    (acc, x, n, p, cam), prev = random_frames(1, W, H, nasty=False)
    bufs = {"accum": acc, "position": x, "normal": n, "prim": p,
            "prev_position": prev["position"], "prev_normal": prev["normal"], "prev_prim": prev["prim"],
            "prev_color": prev["color"], "prev_length": prev["length"],
            "color": np.full((H, W, 4), 7.0, np.float32), "length": np.full((H, W), 7.0, np.float32),
            "pixels": np.full((H, W, 4), 7, np.uint8)}
    return bufs, cam, prev["camera"]


def _untouched(bufs):
    return (bufs["color"] == 7).all() and (bufs["length"] == 7).all() and (bufs["pixels"] == 7).all()


def _call(rt, bufs, cam, pcam, W=8, H=4, spp=4, opt=None, history=True, **over):
    addr = {k: v.ctypes.data for k, v in bufs.items()}
    addr.update(over)
    hist = {}
    if history:
        hist = dict(prev_camera=over.get("prev_camera_floats", pcam), prev_position=addr["prev_position"],
                    prev_normal=addr["prev_normal"], prev_prim=addr["prev_prim"], prev_color=addr["prev_color"],
                    prev_length=addr["prev_length"])
    rt.temporal_accumulate_device(opt if opt is not None else rt.TemporalOptions(), W, H, addr["accum"], spp,
                                  addr["position"], addr["normal"], addr["prim"], over.get("camera_floats", cam),
                                  addr["color"], addr["length"], addr["pixels"], **hist)


BAD_CAM = np.float32([0, 0, 0, -1, -1, -1, 2, 0, 0, 0, np.inf, 0])
REJECTED = [
    ("max_history", dict(opt=dict(max_history=2 ** 20 + 1)), "max_history must be in 1..2^20"),
    ("normal_cos_big", dict(opt=dict(normal_cos=1.5)), "normal_cos must be finite and in [-1, 1]"),
    ("normal_cos_nan", dict(opt=dict(normal_cos=float("nan"))), "normal_cos must be finite and in [-1, 1]"),
    ("plane_tol_negative", dict(opt=dict(plane_tol=-0.1)), "plane_tol must be finite and > 0"),
    ("plane_tol_nan", dict(opt=dict(plane_tol=float("nan"))), "plane_tol must be finite and > 0"),
    ("plane_tol_inf", dict(opt=dict(plane_tol=float("inf"))), "plane_tol must be finite and > 0"),
    ("spp_zero", dict(spp=0), "spp must be >= 1"),
    ("accum_null", dict(over=dict(accum=0)), "the accum buffer is NULL"),
    ("position_null", dict(over=dict(position=0)), "the position buffer is NULL"),
    ("normal_null", dict(over=dict(normal=0)), "the normal buffer is NULL"),
    ("prim_null", dict(over=dict(prim=0)), "the prim buffer is NULL"),
    ("camera_null", dict(camera=None), "the camera is NULL"),
    ("camera_inf", dict(camera=BAD_CAM), "the camera has a non-finite float"),
    ("prev_camera_null", dict(pcam=None), "only partly given: its camera is NULL"),
    ("prev_camera_nan", dict(pcam=np.where(np.arange(12) == 4, np.nan, 1.0).astype(np.float32)),
     "the previous camera has a non-finite float"),
    ("prev_prim_null", dict(over=dict(prev_prim=0)), "only partly given: the previous prim is NULL"),
    ("prev_color_null", dict(over=dict(prev_color=0)), "only partly given: the previous color is NULL"),
    ("prev_length_null", dict(over=dict(prev_length=0)), "only partly given: the previous length is NULL"),
    ("color_null", dict(over=dict(color=0)), "the color output is NULL"),
    ("length_null", dict(over=dict(length=0)), "the length output is NULL"),
    ("width_zero", dict(W=0), "at least 1x1"),
    ("too_tall", dict(H=2 ** 30), "framebuffer too large"),
    ("color_over_prev_color", dict(over="color:prev_color"), "the color output overlaps the previous color input"),
    ("length_over_prev_length", dict(over="length:prev_length"), "the length output overlaps the previous length input"),
    ("pixels_over_accum_tail", dict(over="pixels:accum+"), "the pixels output overlaps the accum input"),
    ("length_over_color", dict(over="length:color"), "the length output overlaps the color output"),
    ("pixels_over_length", dict(over="pixels:length"), "the pixels output overlaps the length output"),
]


@pytest.mark.parametrize("name,spec,text", REJECTED, ids=[r[0] for r in REJECTED])
def test_rejections_fail_on_the_host(rt, name, spec, text):
    bufs, cam, pcam = _host_frame()
    over = spec.get("over", {})
    if isinstance(over, str):                               # "out:in": the output placed on (or into) another buffer
        out, inp = over.split(":")
        tail = inp.endswith("+")
        inp = inp.rstrip("+")
        over = {out: bufs[inp].ctypes.data + (bufs[inp].nbytes - 4 if tail else 0)}
    over = dict(over)
    if "camera" in spec:
        over["camera_floats"] = spec["camera"]
    if "pcam" in spec:
        over["prev_camera_floats"] = spec["pcam"]
    with pytest.raises(rt.RenderError) as e:
        _call(rt, bufs, cam, pcam, W=spec.get("W", 8), H=spec.get("H", 4), spp=spec.get("spp", 4),
              opt=rt.TemporalOptions(**spec.get("opt", {})), **over)
    assert str(e.value).startswith("temporal: ") and text in str(e.value), str(e.value)
    assert _untouched(bufs)


def test_null_options_struct_sizes_guides_and_history_members(rt):
    L = rt.lib()
    bufs, cam, pcam = _host_frame()
    g = rt.AovBuffers(C.sizeof(rt.AovBuffers), 0, None, bufs["position"].ctypes.data, bufs["normal"].ctypes.data, None,
                      bufs["prim"].ctypes.data)
    c12 = (C.c_float * 12)(*cam)
    args = (8, 4, bufs["accum"].ctypes.data, 4)
    outs = (bufs["color"].ctypes.data, bufs["length"].ctypes.data, None, None)
    assert L.rt_temporal_accumulate_device(None, *args, C.byref(g), c12, None, *outs) != 0
    assert "options is NULL" in rt.last_error()
    o = rt.TemporalOptions()._c(None)
    o.struct_size = 24
    assert L.rt_temporal_accumulate_device(C.byref(o), *args, C.byref(g), c12, None, *outs) != 0
    assert "options->struct_size" in rt.last_error()
    o = rt.TemporalOptions()._c(None)
    assert L.rt_temporal_accumulate_device(C.byref(o), *args, None, c12, None, *outs) != 0
    assert "guides is NULL" in rt.last_error()
    pc = (C.c_float * 12)(*pcam)
    pg = rt.AovBuffers(C.sizeof(rt.AovBuffers), 0, None, bufs["prev_position"].ctypes.data,
                       bufs["prev_normal"].ctypes.data, None, bufs["prev_prim"].ctypes.data)
    h = rt._TemporalHistory(C.sizeof(rt._TemporalHistory) - 8, 0, C.cast(pc, C.POINTER(C.c_float)), C.pointer(pg),
                            bufs["prev_color"].ctypes.data, bufs["prev_length"].ctypes.data)
    assert L.rt_temporal_accumulate_device(C.byref(o), *args, C.byref(g), c12, C.byref(h), *outs) != 0
    assert "history->struct_size" in rt.last_error()
    h.struct_size = C.sizeof(rt._TemporalHistory)
    h.guides = None                                          # a history without its guides is only partly given
    assert L.rt_temporal_accumulate_device(C.byref(o), *args, C.byref(g), c12, C.byref(h), *outs) != 0
    assert "only partly given: the previous position is NULL" in rt.last_error()
    empty = rt._TemporalHistory(C.sizeof(rt._TemporalHistory), 0, None, None, None, None)
    assert L.rt_temporal_accumulate_device(C.byref(o), *args, C.byref(g), c12, C.byref(empty), *outs) != 0
    assert "only partly given: its camera is NULL" in rt.last_error()
    assert _untouched(bufs)


def test_valid_call_never_falls_back(rt):
    """A valid call with host arrays fails — without a device because there is none, with one because the arrays are
    not device memory — and never writes an output on the CPU."""
    bufs, cam, pcam = _host_frame()
    for history in (False, True):
        with pytest.raises(rt.RenderError) as e:
            _call(rt, bufs, cam, pcam, history=history)
        want = "no CUDA device available" if rt.device_count() == 0 else "buffer is not device memory of device"
        assert want in str(e.value), str(e.value)
        assert _untouched(bufs)


# ------------------------------------------------------------------------------- device functions on the host

@pytest.fixture(scope="module")
def hostsim():
    subprocess.run(["make", "-C", str(TEMPORAL_HOST), "build/libtemporal_hostsim.so"], check=True, capture_output=True)
    L = C.CDLL(str(TEMPORAL_HOST / "build" / "libtemporal_hostsim.so"))
    L.hostsim_temporal.restype = C.c_int
    L.hostsim_temporal.argtypes = [C.c_uint32, C.c_uint32, C.c_void_p, C.c_int32] + [C.c_void_p] * 10 + \
                                  [C.c_uint32, C.c_float, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p]
    return L


def hostsim_temporal(L, accum, spp, position, normal, prim, camera, prev=None, max_history=0, normal_cos=0.0,
                     plane_tol=0.0):
    H, W = prim.shape
    keep = []

    def a(x, dt=np.float32):
        if x is None:
            return None
        x = np.ascontiguousarray(x, dt)
        keep.append(x)
        return x.ctypes.data

    p = prev or {}
    color, length, pixels = np.zeros((H, W, 4), np.float32), np.zeros((H, W), np.float32), np.zeros((H, W, 4), np.uint8)
    rc = L.hostsim_temporal(W, H, a(accum), spp, a(position), a(normal), a(prim, np.int32), a(camera),
                            a(p.get("camera")), a(p.get("position")), a(p.get("normal")), a(p.get("prim"), np.int32),
                            a(p.get("color")), a(p.get("length")), int(max_history or DEFAULTS["max_history"]),
                            float(normal_cos or DEFAULTS["normal_cos"]), float(plane_tol or DEFAULTS["plane_tol"]),
                            color.ctypes.data, length.ctypes.data, pixels.ctypes.data)
    assert rc == 0
    return {"color": color, "length": length, "pixels": pixels}


@pytest.mark.parametrize("W,H", [(1, 1), (7, 1), (1, 5), (123, 77)])
def test_device_functions_on_host_equal_reference_on_random_frames(hostsim, W, H):
    edges = inside = behind = 0
    for seed in range(4):
        (acc, x, n, p, cam), prev = random_frames(100 * seed + W + H, W, H)
        spp = 1 + seed * 3
        opts = dict(max_history=(0, 5, 1000, 1)[seed], normal_cos=(0.0, 0.5, -1.0, 1.0)[seed],
                    plane_tol=(0.0, 0.05, 0.5, 1e-4)[seed])
        for pv in (None, prev, dict(prev, camera=cam)):                    # no history, reprojection, identity rule
            want = temporal_reference(acc, spp, x, n, p, cam, pv, **opts)
            assert_same(hostsim_temporal(hostsim, acc, spp, x, n, p, cam, pv, **opts), want)
        px, py, ok = project(prev["camera"], x, W, H)
        with np.errstate(invalid="ignore"):
            edges += int(np.sum((px == -1) | (px == W) | (py == -1) | (py == H)))
            inside += int(np.sum(ok))
            behind += int(np.sum(~ok & np.isfinite(px)))
    assert inside > 0 and behind > 0
    if W * H > 1000:                                                       # the border sweep lands exactly on it
        assert edges > 0


def _path_cameras(ob, cam, frames, step=PATH_STEP):
    cams = [cam]
    for _ in range(frames - 1):
        cams.append(ob.move_camera_position(cams[-1], *step))
    return cams


def _oracle_frames(ob, scenes, key, camera, W, H, spp, frames, static=False):
    """Per frame: (sums of spp samples from sample index spp*i, guides at pixel centres, camera floats) along a path
    (or with a static camera)."""
    import test_aov
    cam, world = cases.oracle_scene(ob, scenes, key, camera)
    cams = [cam] * frames if static else _path_cameras(ob, cam, frames)
    out = []
    for i, c in enumerate(cams):
        _, _, accum = ob.ray_trace(world, c, W, H, spp, 8, want_accum=True, sample_begin=spp * i)
        g = test_aov.primary_hits(ob, world, c, W, H, fixed_jitter=True)
        out.append((accum, g, c.floats()))
    return out, world, cams


def _run_path(frames, spp, sim=None, **opts):
    """temporal_reference (and the host build when `sim` is given) along oracle frames; returns the outputs."""
    results, prev = [], None
    for accum, g, cam in frames:
        args = (accum, spp, g["position"], g["normal"], g["prim"], cam, prev)
        out = temporal_reference(*args, **opts)
        if sim is not None:
            assert_same(hostsim_temporal(sim, *args, **opts), out)
        results.append(out)
        prev = {"camera": cam, "position": g["position"], "normal": g["normal"], "prim": g["prim"],
                "color": out["color"], "length": out["length"]}
    return results


@pytest.mark.parametrize("key,camera,W,H,spp", [("default", "file", 160, 90, 4), ("example", "file", 123, 77, 3),
                                                ("c3", "file", 96, 54, 2)])
def test_device_functions_on_host_equal_reference_on_oracle_frames(hostsim, ob, scenes, key, camera, W, H, spp):
    frames, _, _ = _oracle_frames(ob, scenes, key, camera, W, H, spp, 3)
    _run_path(frames, spp, hostsim)
    _run_path(frames, spp, hostsim, max_history=4, normal_cos=0.5, plane_tol=0.1)


# ------------------------------------------------------------------------------------------------ known answers

def test_first_frame_is_the_mean_and_the_oracle_rgba8(ob, scenes):
    W, H, spp = 123, 77, 3
    cam, world = cases.oracle_scene(ob, scenes, "example", "file")
    pixels, _, accum = ob.ray_trace(world, cam, W, H, spp, 8, want_accum=True)
    import test_aov
    g = test_aov.primary_hits(ob, world, cam, W, H, fixed_jitter=True)
    out = temporal_reference(accum, spp, g["position"], g["normal"], g["prim"], cam.floats())
    assert (_bits(out["color"]) == _bits(accum * (f32(1) / f32(spp)))).all()
    assert (out["length"] == f32(spp)).all()
    assert np.array_equal(out["pixels"], pixels)


def test_static_camera_accumulates_like_the_progressive_frame(ob, scenes):
    """k frames of n spp with a static camera (and max_history above k*n): at hit pixels length k*n exactly and rgb
    the k*n-spp mean within a relative 1e-5; a miss pixel (no history by definition) has its last frame's mean."""
    W, H, n, k = 96, 54, 4, 4
    frames, world, cams = _oracle_frames(ob, scenes, "default", "file", W, H, n, k, static=True)
    last = _run_path(frames, n, max_history=1000)[-1]
    _, _, ref = ob.ray_trace(world, cams[0], W, H, n * k, 8, want_accum=True)
    ref = ref * (f32(1) / f32(n * k))
    hit = frames[-1][1]["prim"] >= 0
    assert hit.mean() > 0.5
    assert (last["length"][hit] == f32(n * k)).all() and (last["length"][~hit] == f32(n)).all()
    rgb = (slice(None), slice(0, 3))                                    # the sums' alpha is 1 + spp, not spp
    assert np.allclose(last["color"][hit][rgb], ref[hit][rgb], rtol=1e-5, atol=0)
    assert (_bits(last["color"][~hit]) == _bits(frames[-1][0][~hit] * (f32(1) / f32(n)))).all()


def _tap_rays(pcam, qx, qy, W, H):
    """The previous camera's pixel-centre rays (RtRay records) of previous pixels (qx, qy)."""
    c = np.asarray(pcam, np.float32)
    u = (qx.astype(np.float32) + f32(0.5)) / f32(W - 1)
    t = (f32(H - 1) - qy.astype(np.float32) + f32(0.5)) / f32(H - 1)
    d = ((c[3:6] + c[6:9] * u[:, None]) + c[9:12] * t[:, None]) - c[0:3]
    rays = np.zeros((len(qx), 8), np.float32)
    rays[:, 0:3] = c[0:3]
    rays[:, 3] = np.inf
    rays[:, 4:7] = d
    return rays


def test_disoccluded_pixels_start_over(ob, scenes):
    """Along a camera path, trace (the ray reference) from the previous camera through each of the 2x2 previous pixels
    around a hit pixel's projection.  Where every one of those rays ends at a point more than plane_tol off the pixel's
    tangent plane (an occluder, or the background), the pixel was hidden from the previous camera: it must start over
    with length spp.  Such pixels must exist on the path."""
    import test_rays
    W, H, spp = 160, 90, 4
    frames, world, _ = _oracle_frames(ob, scenes, "default", "file", W, H, spp, 4)
    outs = _run_path(frames, spp)
    found = 0
    for i in range(1, len(frames)):
        _, g, _ = frames[i]
        pcam = frames[i - 1][2]
        X, nrm = g["position"], g["normal"]
        x, y, ok = project(pcam, X, W, H)
        ok &= g["prim"] >= 0
        ys, xs = np.nonzero(ok)
        x0, y0 = np.floor(x[ys, xs]).astype(np.int64), np.floor(y[ys, xs]).astype(np.int64)
        hidden = np.ones(len(ys), bool)
        for dx, dy in ((0, 0), (1, 0), (0, 1), (1, 1)):
            qx, qy = np.clip(x0 + dx, 0, W - 1), np.clip(y0 + dy, 0, H - 1)
            rec = test_rays.reference(ob, world, _tap_rays(pcam, qx, qy, W, H))
            with np.errstate(invalid="ignore"):
                off = np.abs(_dot(nrm[ys, xs], rec["position"] - X[ys, xs])) > f32(DEFAULTS["plane_tol"])
            hidden &= (rec["prim"] < 0) | off
        found += int(hidden.sum())
        assert (outs[i]["length"][ys[hidden], xs[hidden]] == f32(spp)).all()
    assert found > 0


def mse_hits(color, reference, prim):
    hit = prim >= 0
    d = color[..., :3][hit].astype(np.float64) - reference[..., :3][hit].astype(np.float64)
    return float(np.mean(d * d))


def test_quality_along_a_camera_path(ob, scenes):
    """world.txt at 160x90, 8 frames of 4 spp along a camera path: the last frame's error against 1024 spp of the last
    camera is at most half the noisy 4-spp frame's (DESIGN.md §15.4 records the measured ratio)."""
    W, H, spp = 160, 90, 4
    frames, world, cams = _oracle_frames(ob, scenes, "default", "file", W, H, spp, 8)
    last = _run_path(frames, spp)[-1]
    _, _, ref = ob.ray_trace(world, cams[-1], W, H, 1024, 8, want_accum=True, sample_begin=10_000)
    ref = ref / f32(1024)
    prim = frames[-1][1]["prim"]
    e_noisy = mse_hits(frames[-1][0] / f32(spp), ref, prim)
    e_temporal = mse_hits(last["color"], ref, prim)
    assert e_temporal <= 0.5 * e_noisy, (e_temporal, e_noisy)


# ------------------------------------------------------------------------------------------------------------ GPU

def _gpu_frame(gpu_rt, h, W, H, spp, depth=8, sample_begin=0, device=0):
    """accum (torch float32 [H,W,4]) of render_device with RT_OPT_ACCUM_OUT, render_aov's guides (fixed jitter), the
    RGBA8 frame and the camera floats."""
    import torch
    dev = torch.device("cuda", device)
    accum = torch.empty((H, W, 4), dtype=torch.float32, device=dev)
    frame = torch.empty((H, W), dtype=torch.int32, device=dev)
    gpu_rt.render_device(h, gpu_rt.Options(samples_per_pixel=spp, max_ray_bounces=depth, accum_out=True,
                                           sample_begin=sample_begin, device=device),
                         W, H, frame.data_ptr(), accum.data_ptr())
    torch.cuda.synchronize(dev)
    guides = gpu_rt.render_aov(h, W, H, gpu_rt.Options(fixed_jitter=True, device=device))
    return accum, guides, frame, h.camera_floats()


def _np_prev(cam, guides, out):
    return {"camera": cam, "position": guides["position"].cpu().numpy(), "normal": guides["normal"].cpu().numpy(),
            "prim": guides["prim"].cpu().numpy(), "color": out["color"].cpu().numpy(),
            "length": out["length"].cpu().numpy()}


def _gpu_path_against_reference(gpu_rt, h, W, H, spp, depth=8, frames=3, **opts):
    """Frames along a camera path (then one more with the camera standing still), each accumulated on the GPU from the
    GPU's own previous output, against the reference of the same inputs."""
    prev_t, prev_np = None, None
    for i in range(frames + 1):
        if 0 < i < frames:
            gpu_rt.move_camera_position(h, *PATH_STEP)
        accum, g, _, cam = _gpu_frame(gpu_rt, h, W, H, spp, depth, sample_begin=spp * i)
        st = gpu_rt.RenderStats()
        out = gpu_rt.temporal_accumulate(accum, spp, g, cam, prev_t, gpu_rt.TemporalOptions(**opts), stats=st)
        got = {k: v.cpu().numpy() for k, v in out.items()}
        want = temporal_reference(accum.cpu().numpy(), spp, g["position"].cpu().numpy(), g["normal"].cpu().numpy(),
                                  g["prim"].cpu().numpy(), cam, prev_np, **opts)
        assert_same(got, want, canonical_nan=True)
        assert st.launches == 1 and st.rays == 0 and st.samples == 0 and st.kernel_ms > 0
        assert st.total_ms >= st.kernel_ms and st.block == 256 and st.grid > 0
        prev_t = {"camera": cam, "guides": g, "color": out["color"], "length": out["length"]}
        prev_np = _np_prev(cam, g, out)


@pytest.mark.gpu
@pytest.mark.parametrize("case", cases.SMALL_CASES, ids=[c[0] for c in cases.SMALL_CASES])
def test_gpu_small_cases(gpu_rt, scenes, case):
    name, key, camera, W, H, spp, depth, fixed = case
    h = cases.product_scene(gpu_rt, scenes, key, camera)
    _gpu_path_against_reference(gpu_rt, h, W, H, spp, depth)


@pytest.mark.gpu
@pytest.mark.parametrize("W,H", [(1, 1), (7, 1), (1, 5), (123, 77), (1920, 1080)])
def test_gpu_sizes(gpu_rt, scenes, W, H):
    h = gpu_rt.load_world(scenes.example_world())
    _gpu_path_against_reference(gpu_rt, h, W, H, 4, frames=2)


@pytest.mark.gpu
def test_gpu_c3_1080p_and_options(gpu_rt, scenes):
    h = cases.product_scene(gpu_rt, scenes, "c3", "file")
    _gpu_path_against_reference(gpu_rt, h, 1920, 1080, 2, frames=2)
    h = cases.product_scene(gpu_rt, scenes, "c3", "file")
    _gpu_path_against_reference(gpu_rt, h, 320, 180, 2, frames=2, max_history=3, normal_cos=0.5, plane_tol=0.1)


@pytest.mark.gpu
def test_gpu_random_frames_with_nans(gpu_rt):
    import torch
    (acc, x, n, p, cam), prev = random_frames(77, 123, 77)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()   # noqa: E731
    guides = {"position": t(x), "normal": t(n), "prim": t(p)}
    pg = {"position": t(prev["position"]), "normal": t(prev["normal"]), "prim": t(prev["prim"])}
    for pv in (prev, dict(prev, camera=cam)):
        prev_t = {"camera": pv["camera"], "guides": pg, "color": t(prev["color"]), "length": t(prev["length"])}
        got = gpu_rt.temporal_accumulate(t(acc), 3, guides, cam, prev_t, gpu_rt.TemporalOptions(plane_tol=0.05))
        want = temporal_reference(acc, 3, x, n, p, cam, pv, plane_tol=0.05)
        assert_same({k: v.cpu().numpy() for k, v in got.items()}, want, canonical_nan=True)


@pytest.mark.gpu
def test_gpu_first_frame_pixels_equal_the_render(gpu_rt, scenes):
    h = gpu_rt.load_world(scenes.default_world())
    W, H = 320, 180
    accum, g, frame, cam = _gpu_frame(gpu_rt, h, W, H, 8)
    out = gpu_rt.temporal_accumulate(accum, 8, g, cam)
    assert np.array_equal(out["pixels"].cpu().numpy(), frame.cpu().numpy().view(np.uint8).reshape(H, W, 4))
    assert (out["length"] == 8).all()


@pytest.mark.gpu
def test_gpu_temporal_renderer_static_camera_and_denoise(gpu_rt, scenes):
    """A static camera: k frames of n spp give, at hit pixels, length k*n and the k*n-spp progressive mean within a
    relative 1e-5; the denoised output is denoise(color, 1, guides) of the accumulation."""
    import torch
    W, H, n, k = 320, 180, 4, 5
    h = gpu_rt.load_world(scenes.default_world())
    r = gpu_rt.TemporalRenderer(W, H, gpu_rt.Options(samples_per_pixel=n), gpu_rt.TemporalOptions(max_history=1000),
                                gpu_rt.DenoiseOptions())
    for _ in range(k):
        out = r.frame(h)
    ref = torch.empty((H, W, 4), dtype=torch.float32, device="cuda")
    px = torch.empty((H, W), dtype=torch.int32, device="cuda")
    gpu_rt.render_device(h, gpu_rt.Options(samples_per_pixel=n * k, accum_out=True), W, H, px.data_ptr(), ref.data_ptr())
    torch.cuda.synchronize()
    mean = ref.cpu().numpy() * (f32(1) / f32(n * k))
    guides = gpu_rt.render_aov(h, W, H, gpu_rt.Options(fixed_jitter=True))
    hit = guides["prim"].cpu().numpy() >= 0
    assert (out["length"].cpu().numpy()[hit] == n * k).all()
    assert np.allclose(out["color"].cpu().numpy()[hit][:, :3], mean[hit][:, :3], rtol=1e-5, atol=0)
    by_hand = gpu_rt.denoise(out["color"], 1, guides)
    for key in ("pixels", "color"):
        assert np.array_equal(_bits(out["denoised"][key].cpu().numpy(), True), _bits(by_hand[key].cpu().numpy(), True))
    # a camera move keeps part of the history; reset() and a resize drop all of it
    gpu_rt.move_camera_position(h, *PATH_STEP)
    moved = r.frame(h)["length"].cpu().numpy()
    assert (moved > n).mean() > 0.5 and (moved == n).any()
    r.reset()
    assert (r.frame(h)["length"] == n).all()
    assert (r.frame(h)["length"] > n).any()
    r.width, r.height = 160, 90
    assert (r.frame(h)["length"] == n).all()


@pytest.mark.gpu
def test_gpu_outputs_stream_device_and_stats(gpu_rt, scenes):
    import torch
    h = gpu_rt.load_world(scenes.c3_world())
    W, H = 320, 180
    a0, g0, _, c0 = _gpu_frame(gpu_rt, h, W, H, 4)
    gpu_rt.move_camera_position(h, *PATH_STEP)
    a1, g1, _, c1 = _gpu_frame(gpu_rt, h, W, H, 4, sample_begin=4)
    np0 = [t.cpu().numpy() for t in (a0, g0["position"], g0["normal"], g0["prim"])]
    np1 = [t.cpu().numpy() for t in (a1, g1["position"], g1["normal"], g1["prim"])]
    want0 = temporal_reference(*np0[:1], 4, *np0[1:], c0)
    prev_np = {"camera": c0, "position": np0[1], "normal": np0[2], "prim": np0[3], "color": want0["color"],
               "length": want0["length"]}
    want1 = temporal_reference(*np1[:1], 4, *np1[1:], c1, prev_np)
    ptr = lambda g: (g["position"].data_ptr(), g["normal"].data_ptr(), g["prim"].data_ptr())   # noqa: E731

    def outs():                                          # filled before the library's own stream writes them
        o = (torch.full((H, W, 4), 7.0, device="cuda"), torch.full((H, W), 7.0, device="cuda"),
             torch.full((H, W, 4), 7, dtype=torch.uint8, device="cuda"))
        torch.cuda.synchronize()
        return o

    # the optional output alone is left out; the required ones alone
    col, ln, px = outs()
    gpu_rt.temporal_accumulate_device(None, W, H, a0.data_ptr(), 4, *ptr(g0), c0, col.data_ptr(), ln.data_ptr())
    assert_same({"color": col.cpu().numpy(), "length": ln.cpu().numpy()}, want0, canonical_nan=True)
    assert (px == 7).all()
    # two chained frames ordered on a caller's stream behind a busy kernel: the calls return once enqueued
    s = torch.cuda.Stream()
    c_a, l_a, p_a = outs()
    c_b, l_b, p_b = outs()
    torch.cuda.synchronize()
    with torch.cuda.stream(s):
        torch.cuda._sleep(200_000_000)
    gpu_rt.temporal_accumulate_device(gpu_rt.TemporalOptions(device=0), W, H, a0.data_ptr(), 4, *ptr(g0), c0,
                                      c_a.data_ptr(), l_a.data_ptr(), p_a.data_ptr(), stream=s.cuda_stream)
    gpu_rt.temporal_accumulate_device(None, W, H, a1.data_ptr(), 4, *ptr(g1), c1, c_b.data_ptr(), l_b.data_ptr(),
                                      p_b.data_ptr(), prev_camera=c0, prev_position=g0["position"].data_ptr(),
                                      prev_normal=g0["normal"].data_ptr(), prev_prim=g0["prim"].data_ptr(),
                                      prev_color=c_a.data_ptr(), prev_length=l_a.data_ptr(), stream=s.cuda_stream)
    assert not s.query(), "the calls waited for the caller's stream"
    s.synchronize()
    assert_same({"color": c_a.cpu().numpy(), "length": l_a.cpu().numpy(), "pixels": p_a.cpu().numpy()}, want0,
                canonical_nan=True)
    assert_same({"color": c_b.cpu().numpy(), "length": l_b.cpu().numpy(), "pixels": p_b.cpu().numpy()}, want1,
                canonical_nan=True)
    # stats on a caller's stream wait for the kernel time
    st = gpu_rt.RenderStats()
    c_c, l_c, _ = outs()
    with torch.cuda.stream(s):
        torch.cuda._sleep(50_000_000)
    gpu_rt.temporal_accumulate_device(None, W, H, a0.data_ptr(), 4, *ptr(g0), c0, c_c.data_ptr(), l_c.data_ptr(),
                                      stream=s.cuda_stream, stats=st)
    assert s.query() and st.kernel_ms > 0 and st.launches == 1 and st.block == 256
    assert st.grid == ((W + 31) // 32) * ((H + 7) // 8)
    # `device` names a device explicitly (the last one); the caller's current device is left as it was
    n = torch.cuda.device_count()
    target = n - 1
    torch.cuda.set_device(0)
    hd = gpu_rt.load_world(scenes.c3_world())
    a_d, g_d, _, c_d = _gpu_frame(gpu_rt, hd, W, H, 4, device=target)
    col = torch.full((H, W, 4), 7.0, device=f"cuda:{target}")
    ln = torch.full((H, W), 7.0, device=f"cuda:{target}")
    torch.cuda.synchronize(target)
    gpu_rt.temporal_accumulate_device(gpu_rt.TemporalOptions(device=target), W, H, a_d.data_ptr(), 4, *ptr(g_d), c_d,
                                      col.data_ptr(), ln.data_ptr())
    assert torch.cuda.current_device() == 0
    npd = [t.cpu().numpy() for t in (a_d, g_d["position"], g_d["normal"], g_d["prim"])]
    assert_same({"color": col.cpu().numpy(), "length": ln.cpu().numpy()},
                temporal_reference(*npd[:1], 4, *npd[1:], c_d), canonical_nan=True)
