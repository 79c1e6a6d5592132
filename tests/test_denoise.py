"""Denoiser (rt_denoise_device / denoise / render_denoised): the edge-avoiding a-trous filter of a frame's colour sums,
guided by the first-hit buffers, equal to the numpy reference below bit for bit.

`denoise_reference` restates DESIGN.md §12.1 in numpy float32, vectorised over pixels, with a Python loop over the
iterations and the 25 taps in the kernel's order.  A skipped tap adds +0.0 to the sums, which leaves them unchanged
(they start at +0.0 and so are never -0.0), so the masked sum equals the kernel's branchy one.

CPU tests: the boundary (symbols, struct layout, every rejection), known answers of the reference, the device header's
per-pixel functions built for the host (tests/denoise_host) against the reference, and the quality on an oracle frame.
GPU tests: the kernel against the reference on frames the library renders.  Between the GPU and the CPU a NaN is
compared as "NaN" (IEEE leaves a generated NaN's sign and payload to the hardware).
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
DENOISE_HOST = HERE / "denoise_host"
f32 = np.float32
TAPS = np.array([1 / 16, 1 / 4, 3 / 8, 1 / 4, 1 / 16], np.float32)          # §1 h[-2..2]
FLOOR = f32(2.0 ** -10)                                                      # §1 a' = max(albedo, 2^-10)
DEFAULTS = {"iterations": 5, "sigma_color": 1.0, "sigma_normal": 0.25, "sigma_plane": 0.02}


# ------------------------------------------------------------------------------------------------------- reference

def scale(sigma):
    """§1: 1 / ((16 sigma) sigma) in float32."""
    s = f32(sigma)
    return f32(1) / ((f32(16) * s) * s)


def _dot(a, b):
    """§1: (a.x*b.x + a.y*b.y) + a.z*b.z"""
    return (a[..., 0] * b[..., 0] + a[..., 1] * b[..., 1]) + a[..., 2] * b[..., 2]


def _shift(a, ox, oy):
    """a[y + oy, x + ox] at every (y, x), and where that is inside the frame."""
    H, W = a.shape[:2]
    out = np.zeros_like(a)
    ok = np.zeros((H, W), bool)
    y0, y1, x0, x1 = max(0, -oy), min(H, H - oy), max(0, -ox), min(W, W - ox)
    if y0 < y1 and x0 < x1:
        out[y0:y1, x0:x1] = a[y0 + oy:y1 + oy, x0 + ox:x1 + ox]
        ok[y0:y1, x0:x1] = True
    return out, ok


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


def denoise_reference(accum, spp, normal, position, albedo, prim, iterations=0, sigma_color=0.0, sigma_normal=0.0,
                      sigma_plane=0.0):
    """{"color": float32 [H,W,4], "pixels": uint8 [H,W,4]} of DESIGN.md §12.1; a 0 option takes its default."""
    accum, normal, position, albedo = (np.asarray(a, np.float32) for a in (accum, normal, position, albedo))
    n_it = int(iterations) or DEFAULTS["iterations"]
    sc = scale(sigma_color or DEFAULTS["sigma_color"])
    sn = scale(sigma_normal or DEFAULTS["sigma_normal"])
    sx = scale(sigma_plane or DEFAULTS["sigma_plane"])
    with np.errstate(all="ignore"):
        m = accum * (f32(1) / f32(spp))                                      # mean, alpha included
        miss = np.asarray(prim) < 0                                          # pixel classes
        a = np.fmax(albedo, FLOOR)                                           # demodulation (fmaxf: NaN -> 2^-10)
        e = m[..., :3] / a
        for i in range(n_it):                                                # iteration i: step 2^i
            s, sc_i = 1 << i, sc * f32(4 ** i)
            sw = np.zeros(miss.shape, np.float32)
            acc = np.zeros(e.shape, np.float32)
            for dy in range(-2, 3):                                          # tap order: dy outer, dx inner
                for dx in range(-2, 3):
                    eq, inside = _shift(e, dx * s, dy * s)
                    nq, _ = _shift(normal, dx * s, dy * s)
                    xq, _ = _shift(position, dx * s, dy * s)
                    mq, _ = _shift(miss, dx * s, dy * s)
                    dc, dn = e - eq, normal - nq
                    uc = _dot(dc, dc) * sc_i                                 # colour term
                    un = _dot(dn, dn) * sn                                   # normal term
                    d = _dot(normal, xq - position)
                    ux = (d * d) * sx                                        # plane-distance term
                    r = f32(1) / (((f32(1) + uc) * (f32(1) + un)) * (f32(1) + ux))
                    for _ in range(4):
                        r = r * r                                            # r^16
                    w = (TAPS[dx + 2] * TAPS[dy + 2]) * r
                    ok = inside & ~mq & (w > 0)                              # skipped taps add +0.0
                    sw = sw + np.where(ok, w, f32(0))
                    acc = acc + np.where(ok[..., None], w[..., None] * eq, f32(0))
            e = np.where((sw > 0)[..., None], acc / sw[..., None], e)        # no accepted tap: unchanged
        color = m.copy()
        color[..., :3] = np.where(miss[..., None], m[..., :3], e * a)       # remodulation; misses get m
    return {"color": color, "pixels": rgba8(color)}


def _bits(a, canonical_nan=False):
    a = np.ascontiguousarray(a)
    if a.dtype != np.float32:
        return a
    b = a.view(np.uint32).copy()
    if canonical_nan:
        b[np.isnan(a)] = 0x7FFFFFFF
    return b


def assert_same(got, want, canonical_nan=False):
    for k in ("color", "pixels"):
        if k not in got:
            continue
        g, w = np.asarray(got[k]), np.asarray(want[k])
        bad = np.argwhere(_bits(g, canonical_nan) != _bits(w, canonical_nan))
        assert bad.size == 0, f"{k}: {len(bad)} values differ, first at {bad[0].tolist()}: {g[tuple(bad[0])]} vs {w[tuple(bad[0])]}"


def random_frame(seed, W, H, nasty=True):
    """Random sums and guides; with `nasty`: zero albedo, misses, NaN guides, NaN and inf sums."""
    rng = np.random.default_rng(seed)
    accum = (rng.random((H, W, 4)) * 8).astype(np.float32)
    normal = rng.normal(size=(H, W, 3)).astype(np.float32)
    normal /= np.linalg.norm(normal, axis=-1, keepdims=True).astype(np.float32)
    normal[rng.random((H, W)) < 0.5] = normal[0, 0]                         # large flat regions
    position = (rng.random((H, W, 3)) * 2).astype(np.float32)
    albedo = rng.random((H, W, 3)).astype(np.float32)
    prim = rng.integers(0, 5, (H, W)).astype(np.int32)
    if nasty:
        albedo[rng.random((H, W)) < 0.05] = 0.0
        albedo[rng.random((H, W)) < 0.02, 1] = np.nan
        prim[rng.random((H, W)) < 0.1] = -1
        normal[rng.random((H, W)) < 0.01] = np.nan
        position[rng.random((H, W)) < 0.01, 2] = np.nan
        accum[rng.random((H, W)) < 0.01, 0] = np.nan
        accum[rng.random((H, W)) < 0.005, 2] = np.inf
    return accum, normal, position, albedo, prim


# ---------------------------------------------------------------------------------------------------------- C ABI

def test_header_declares_the_call_and_the_package_exports_it(rt, tmp_path):
    text = (ROOT / "include" / "raytracer_b200.h").read_text()
    assert "int rt_denoise_device(" in text and "typedef struct RtDenoiseOptions" in text
    assert "rt_denoise_device" in rt.EXPORTED_SYMBOLS and hasattr(rt.lib(), "rt_denoise_device")
    assert rt.lib().rt_abi_version() == 2
    src = tmp_path / "layout.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "raytracer_b200.h"\n'
                   "int main(void) { printf(\"%zu %zu %zu %zu\\n\", sizeof(RtDenoiseOptions), "
                   "offsetof(RtDenoiseOptions, sigma_plane), offsetof(RtDenoiseOptions, device), "
                   "offsetof(RtDenoiseOptions, stats)); return 0; }\n")
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-std=c11", "-I", str(ROOT / "include"), str(src), "-o", str(exe)], check=True)
    size, plane, device, stats = map(int, subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split())
    o = rt._DenoiseOptions
    assert (C.sizeof(o), o.sigma_plane.offset, o.device.offset, o.stats.offset) == (size, plane, device, stats)


def test_defaults_agree_everywhere(rt):
    """The header's RT_DENOISE_DEFAULT_*, the host layer's constants, the package's and this reference's."""
    hdr = (ROOT / "include" / "raytracer_b200.h").read_text()
    host = (ROOT / "rust-swift-raytracer_b200" / "csrc" / "rt_host.hpp").read_text()
    for key, name, cname in (("iterations", "ITERATIONS", "Iterations"), ("sigma_color", "SIGMA_COLOR", "SigmaColor"),
                             ("sigma_normal", "SIGMA_NORMAL", "SigmaNormal"), ("sigma_plane", "SIGMA_PLANE", "SigmaPlane")):
        h = re.search(r"#define RT_DENOISE_DEFAULT_%s ([0-9.]+)[uf]" % name, hdr).group(1)
        c = re.search(r"kDenoiseDefault%s\s*=\s*([0-9.]+)[uf];" % cname, host).group(1)
        assert f32(h) == f32(c) == f32(getattr(rt, "DENOISE_DEFAULT_" + name)) == f32(DEFAULTS[key]), key


def _host_frame(W=8, H=4):
    acc, n, x, a, p = random_frame(1, W, H, nasty=False)
    return {"accum": acc, "normal": n, "position": x, "albedo": a, "prim": p,
            "pixels": np.full((H, W, 4), 7, np.uint8), "color": np.full((H, W, 4), 7.0, np.float32)}


def _call(rt, bufs, W=8, H=4, spp=4, opt=None, which=("pixels", "color"), **over):
    addr = {k: (v.ctypes.data if isinstance(v, np.ndarray) else v) for k, v in bufs.items()}
    addr.update(over)
    rt.denoise_device(opt if opt is not None else rt.DenoiseOptions(), W, H, addr["accum"], spp, addr["normal"],
                      addr["position"], addr["albedo"], addr["prim"], addr["pixels"] if "pixels" in which else 0,
                      addr["color"] if "color" in which else 0)


def _untouched(bufs):
    return (bufs["pixels"] == 7).all() and (bufs["color"] == 7).all()


REJECTED = [
    ("iterations", dict(opt=dict(iterations=11)), "iterations must be in 1..10"),
    ("sigma_negative", dict(opt=dict(sigma_color=-1.0)), "sigma_color must be finite and > 0"),
    ("sigma_nan", dict(opt=dict(sigma_normal=float("nan"))), "sigma_normal must be finite and > 0"),
    ("sigma_inf", dict(opt=dict(sigma_plane=float("inf"))), "sigma_plane must be finite and > 0"),
    ("spp_zero", dict(spp=0), "spp must be >= 1"),
    ("spp_negative", dict(spp=-3), "spp must be >= 1"),
    ("accum_null", dict(over=dict(accum=0)), "the accum buffer is NULL"),
    ("normal_null", dict(over=dict(normal=0)), "the normal buffer is NULL"),
    ("position_null", dict(over=dict(position=0)), "the position buffer is NULL"),
    ("albedo_null", dict(over=dict(albedo=0)), "the albedo buffer is NULL"),
    ("prim_null", dict(over=dict(prim=0)), "the prim buffer is NULL"),
    ("no_outputs", dict(which=()), "both outputs (pixels, color) are NULL"),
    ("width_zero", dict(W=0), "at least 1x1"),
    ("height_zero", dict(H=0), "at least 1x1"),
    ("too_wide", dict(W=2 ** 30), "framebuffer too large"),
    ("pixels_over_accum", dict(over="pixels:accum"), "the pixels output overlaps the accum input"),
    ("color_over_prim", dict(over="color:prim"), "the color output overlaps the prim input"),
    ("color_over_albedo_tail", dict(over="color:albedo+"), "the color output overlaps the albedo input"),
    ("outputs_overlap", dict(over="pixels:color"), "the two outputs overlap"),
]


@pytest.mark.parametrize("name,spec,text", REJECTED, ids=[r[0] for r in REJECTED])
def test_rejections_fail_on_the_host(rt, name, spec, text):
    bufs = _host_frame()
    over = spec.get("over", {})
    if isinstance(over, str):                               # "out:in": the output placed on (or into) an input's bytes
        out, inp = over.split(":")
        tail = inp.endswith("+")
        inp = inp.rstrip("+")
        over = {out: bufs[inp].ctypes.data + (bufs[inp].nbytes - 4 if tail else 0)}
    opt = rt.DenoiseOptions(**spec.get("opt", {}))
    with pytest.raises(rt.RenderError) as e:
        _call(rt, bufs, W=spec.get("W", 8), H=spec.get("H", 4), spp=spec.get("spp", 4), opt=opt,
              which=spec.get("which", ("pixels", "color")), **over)
    assert str(e.value).startswith("denoise: ") and text in str(e.value), str(e.value)
    assert _untouched(bufs)


def test_null_options_struct_size_and_guides(rt):
    L = rt.lib()
    bufs = _host_frame()
    g = rt.AovBuffers(C.sizeof(rt.AovBuffers), 0, None, bufs["position"].ctypes.data, bufs["normal"].ctypes.data,
                      bufs["albedo"].ctypes.data, bufs["prim"].ctypes.data)
    args = (8, 4, bufs["accum"].ctypes.data, 4)
    outs = (bufs["pixels"].ctypes.data, bufs["color"].ctypes.data, None)
    assert L.rt_denoise_device(None, *args, C.byref(g), *outs) != 0
    assert "options is NULL" in rt.last_error()
    o = rt.DenoiseOptions()._c(None)
    o.struct_size = 24
    assert L.rt_denoise_device(C.byref(o), *args, C.byref(g), *outs) != 0
    assert "struct_size" in rt.last_error()
    o = rt.DenoiseOptions()._c(None)
    assert L.rt_denoise_device(C.byref(o), *args, None, *outs) != 0
    assert "guides is NULL" in rt.last_error()
    assert _untouched(bufs)


def test_valid_call_never_falls_back(rt):
    """A valid call with host arrays fails — without a device because there is none, with one because the arrays are
    not device memory — and never writes an output on the CPU."""
    bufs = _host_frame()
    with pytest.raises(rt.RenderError) as e:
        _call(rt, bufs, opt=rt.DenoiseOptions(iterations=3, sigma_color=1.0))
    want = "no CUDA device available" if rt.device_count() == 0 else "buffer is not device memory of device"
    assert want in str(e.value), str(e.value)
    assert _untouched(bufs)


# ------------------------------------------------------------------------------------- known answers of the reference

def _flat(W, H, color=(0.3, 0.6, 0.9, 1.0), spp=4):
    accum = np.broadcast_to(np.float32(color) * f32(spp), (H, W, 4)).astype(np.float32)
    normal = np.broadcast_to(np.float32([0, 1, 0]), (H, W, 3)).astype(np.float32)
    position = np.zeros((H, W, 3), np.float32)
    position[..., 0] = np.arange(W, dtype=np.float32)[None, :] * f32(0.01)
    position[..., 2] = np.arange(H, dtype=np.float32)[:, None] * f32(0.01)
    albedo = np.broadcast_to(np.float32([0.5, 0.25, 0.8]), (H, W, 3)).astype(np.float32)
    return accum, normal, position, albedo, np.zeros((H, W), np.int32)


def test_reference_constant_frame_is_unchanged():
    accum, normal, position, albedo, prim = _flat(37, 23)
    want = accum / f32(4)
    for it in (1, 5, 10):
        got = denoise_reference(accum, 4, normal, position, albedo, prim, iterations=it)["color"]
        ulp = np.abs(got.view(np.int32) - want.view(np.int32))
        assert ulp.max() <= 2, (it, ulp.max())


def test_reference_misses_pass_through_bit_exactly():
    accum, normal, position, albedo, prim = random_frame(3, 40, 30)
    miss = prim < 0
    out = denoise_reference(accum, 7, normal, position, albedo, prim)
    m = accum * (f32(1) / f32(7))
    assert miss.any()
    assert (_bits(out["color"][miss]) == _bits(m[miss])).all()


def test_reference_orthogonal_half_planes_keep_their_colours():
    """Left half: normal +x, colour A; right half: normal +y, colour B.  Across the edge un = |n_p - n_q|^2 sn = 2 sn,
    so every cross-edge tap has r <= 1 / (1 + 2 sn) while its kernel weight is at most 9/64 of the centre's.  The leak
    into a pixel is bounded by the cross-edge share of its weights times |A - B|, and that bound is checked."""
    W, H = 32, 16
    accum, normal, position, albedo, prim = _flat(W, H, spp=1)
    left = np.arange(W)[None, :] < W // 2
    A, B = np.float32([0.9, 0.1, 0.1]), np.float32([0.1, 0.1, 0.9])
    accum[..., :3] = np.where(left[..., None], A, B)
    normal[:] = np.where(left[..., None], np.float32([1, 0, 0]), np.float32([0, 1, 0]))
    albedo[:] = 1.0
    position[:] = 0.0                                                     # plane term 0: only the normal stops the filter
    out = denoise_reference(accum, 1, normal, position, albedo, prim)["color"][..., :3]
    r16 = (1.0 / (1.0 + 2.0 * float(scale(DEFAULTS["sigma_normal"])))) ** 16
    # a pixel's own-side weights sum to at least the centre tap 9/64; at most 24 cross-edge taps of h <= 9/64 each
    share = 24 * (9 / 64) * r16 / (9 / 64 + 24 * (9 / 64) * r16)
    bound = share * np.abs(A - B).max() * 1.0001 + 1e-6
    err = np.abs(out - np.where(left[..., None], A, B)).max()
    assert err <= bound, (err, bound)
    assert bound < 0.05


def test_reference_zero_options_select_the_defaults(rt):
    """The C struct path: DenoiseOptions() carries zeros, which the library replaces by RT_DENOISE_DEFAULT_*; the
    reference does the same, and the result equals the one with the defaults spelled out."""
    o = rt.DenoiseOptions()._c(None)
    assert (o.iterations, o.sigma_color, o.sigma_normal, o.sigma_plane, o.device) == (0, 0.0, 0.0, 0.0, -1)
    frame = random_frame(5, 29, 17)
    a = denoise_reference(*frame[:1], 3, *frame[1:])
    b = denoise_reference(*frame[:1], 3, *frame[1:], iterations=rt.DENOISE_DEFAULT_ITERATIONS,
                          sigma_color=rt.DENOISE_DEFAULT_SIGMA_COLOR, sigma_normal=rt.DENOISE_DEFAULT_SIGMA_NORMAL,
                          sigma_plane=rt.DENOISE_DEFAULT_SIGMA_PLANE)
    assert_same(a, b)
    c = denoise_reference(*frame[:1], 3, *frame[1:], sigma_color=2.0)
    assert not np.array_equal(_bits(a["color"]), _bits(c["color"]))


# ------------------------------------------------------------------------------- device functions on the host

@pytest.fixture(scope="module")
def hostsim():
    subprocess.run(["make", "-C", str(DENOISE_HOST), "build/libdenoise_hostsim.so"], check=True, capture_output=True)
    L = C.CDLL(str(DENOISE_HOST / "build" / "libdenoise_hostsim.so"))
    L.hostsim_denoise.restype = C.c_int
    L.hostsim_denoise.argtypes = [C.c_uint32, C.c_uint32, C.c_void_p, C.c_int32] + [C.c_void_p] * 4 + \
                                 [C.c_uint32, C.c_float, C.c_float, C.c_float, C.c_void_p, C.c_void_p]
    return L


def hostsim_denoise(L, accum, spp, normal, position, albedo, prim, iterations=0, sigma_color=0.0, sigma_normal=0.0,
                    sigma_plane=0.0):
    H, W = prim.shape
    arrs = [np.ascontiguousarray(a) for a in (accum, normal, position, albedo)] + [np.ascontiguousarray(prim, np.int32)]
    pixels = np.zeros((H, W, 4), np.uint8)
    color = np.zeros((H, W, 4), np.float32)
    rc = L.hostsim_denoise(W, H, arrs[0].ctypes.data, spp, *(a.ctypes.data for a in arrs[1:]),
                           int(iterations) or DEFAULTS["iterations"], scale(sigma_color or DEFAULTS["sigma_color"]),
                           scale(sigma_normal or DEFAULTS["sigma_normal"]), scale(sigma_plane or DEFAULTS["sigma_plane"]),
                           pixels.ctypes.data, color.ctypes.data)
    assert rc == 0
    return {"color": color, "pixels": pixels}


@pytest.mark.parametrize("W,H", [(1, 1), (7, 1), (1, 5), (123, 77)])
@pytest.mark.parametrize("iterations", [1, 5, 10])
def test_device_functions_on_host_equal_reference_on_random_frames(hostsim, W, H, iterations):
    for seed in range(3):
        frame = random_frame(100 * seed + W + H, W, H)
        spp = 1 + seed * 5
        opts = dict(iterations=iterations, sigma_color=(0.0, 0.2, 3.0)[seed], sigma_plane=(0.0, 0.5, 0.01)[seed])
        want = denoise_reference(frame[0], spp, *frame[1:], **opts)
        assert_same(hostsim_denoise(hostsim, frame[0], spp, *frame[1:], **opts), want)


def _oracle_frame(ob, scenes, key, camera, W, H, spp, seed=None):
    """Sums of the oracle's render (accum_out) and the guides of the first-hit reference (fixed jitter, sample 0)."""
    import test_aov
    cam, world = cases.oracle_scene(ob, scenes, key, camera)
    kw = {} if seed is None else {"seed": seed}
    _, _, accum = ob.ray_trace(world, cam, W, H, spp, 8, want_accum=True, **kw)
    g = test_aov.primary_hits(ob, world, cam, W, H, fixed_jitter=True, **kw)
    return accum, g["normal"], g["position"], g["albedo"], g["prim"]


@pytest.mark.parametrize("key,camera,W,H,spp", [("default", "file", 160, 90, 4), ("example", "file", 123, 77, 3),
                                                ("c3", "file", 96, 54, 2)])
def test_device_functions_on_host_equal_reference_on_oracle_frames(hostsim, ob, scenes, key, camera, W, H, spp):
    frame = _oracle_frame(ob, scenes, key, camera, W, H, spp)
    for it in (1, 5):
        assert_same(hostsim_denoise(hostsim, frame[0], spp, *frame[1:], iterations=it),
                    denoise_reference(frame[0], spp, *frame[1:], iterations=it))


def mse_hits(color, reference, prim):
    hit = prim >= 0
    d = color[..., :3][hit].astype(np.float64) - reference[..., :3][hit].astype(np.float64)
    return float(np.mean(d * d))


def test_quality_on_an_oracle_frame(ob, scenes):
    """world.txt at 160x90: the denoised 4-spp frame's error against 1024 spp is at most half the noisy frame's."""
    W, H = 160, 90
    frame = _oracle_frame(ob, scenes, "default", "file", W, H, 4)
    cam, world = cases.oracle_scene(ob, scenes, "default", "file")
    _, _, ref = ob.ray_trace(world, cam, W, H, 1024, 8, want_accum=True)
    ref = ref / f32(1024)
    noisy = frame[0] / f32(4)
    den = denoise_reference(frame[0], 4, *frame[1:])["color"]
    e_noisy, e_den = mse_hits(noisy, ref, frame[4]), mse_hits(den, ref, frame[4])
    assert e_den <= 0.5 * e_noisy, (e_den, e_noisy)


# ------------------------------------------------------------------------------------------------------------ GPU

def _gpu_inputs(gpu_rt, h, W, H, spp, depth=8, device=0):
    """accum (torch float32 [H,W,4]) of render_device with RT_OPT_ACCUM_OUT, and render_aov's guides (fixed jitter)."""
    import torch
    dev = torch.device("cuda", device)
    accum = torch.empty((H, W, 4), dtype=torch.float32, device=dev)
    frame = torch.empty((H, W), dtype=torch.int32, device=dev)
    gpu_rt.render_device(h, gpu_rt.Options(samples_per_pixel=spp, max_ray_bounces=depth, accum_out=True, device=device),
                         W, H, frame.data_ptr(), accum.data_ptr())
    torch.cuda.synchronize(dev)
    guides = gpu_rt.render_aov(h, W, H, gpu_rt.Options(fixed_jitter=True, device=device))
    return accum, guides, frame


def _np(inputs):
    accum, g, _ = inputs
    return [accum.cpu().numpy()] + [g[k].cpu().numpy() for k in ("normal", "position", "albedo", "prim")]


def _gpu_denoise(gpu_rt, accum, spp, guides, **opt):
    st = gpu_rt.RenderStats()
    out = gpu_rt.denoise(accum, spp, guides, gpu_rt.DenoiseOptions(**opt), stats=st)
    return {k: v.cpu().numpy() for k, v in out.items()}, st


@pytest.mark.gpu
@pytest.mark.parametrize("case", cases.SMALL_CASES, ids=[c[0] for c in cases.SMALL_CASES])
def test_gpu_small_cases(gpu_rt, scenes, case):
    name, key, camera, W, H, spp, depth, fixed = case
    h = cases.product_scene(gpu_rt, scenes, key, camera)
    inputs = _gpu_inputs(gpu_rt, h, W, H, spp, depth)
    arrs = _np(inputs)
    for it in (1, 5, 10):
        got, st = _gpu_denoise(gpu_rt, inputs[0], spp, inputs[1], iterations=it)
        assert_same(got, denoise_reference(arrs[0], spp, *arrs[1:], iterations=it), canonical_nan=True)
        assert st.launches == 1 + it and st.rays == 0 and st.samples == 0 and st.kernel_ms > 0
        assert st.total_ms >= st.kernel_ms and st.block > 0 and st.grid > 0


@pytest.mark.gpu
@pytest.mark.parametrize("W,H", [(1, 1), (7, 1), (1, 5), (123, 77), (1920, 1080)])
def test_gpu_sizes(gpu_rt, scenes, W, H):
    h = gpu_rt.load_world(scenes.example_world())
    inputs = _gpu_inputs(gpu_rt, h, W, H, 4)
    arrs = _np(inputs)
    for it in ((1, 5, 10) if W * H < 100000 else (5,)):
        got, _ = _gpu_denoise(gpu_rt, inputs[0], 4, inputs[1], iterations=it)
        assert_same(got, denoise_reference(arrs[0], 4, *arrs[1:], iterations=it), canonical_nan=True)


@pytest.mark.gpu
@pytest.mark.parametrize("key,W,H,spp", [("c3", 1920, 1080, 4), ("c5", 1280, 720, 2)])
def test_gpu_large_worlds(gpu_rt, scenes, key, W, H, spp):
    h = cases.product_scene(gpu_rt, scenes, key, "file")
    inputs = _gpu_inputs(gpu_rt, h, W, H, spp)
    arrs = _np(inputs)
    got, _ = _gpu_denoise(gpu_rt, inputs[0], spp, inputs[1])
    assert_same(got, denoise_reference(arrs[0], spp, *arrs[1:]), canonical_nan=True)


@pytest.mark.gpu
def test_gpu_random_inputs_with_nans(gpu_rt):
    import torch
    frame = random_frame(77, 123, 77)
    t = [torch.from_numpy(a).cuda() for a in frame]
    guides = {"normal": t[1], "position": t[2], "albedo": t[3], "prim": t[4]}
    for it in (1, 5, 10):
        got, _ = _gpu_denoise(gpu_rt, t[0], 3, guides, iterations=it, sigma_color=0.7)
        assert_same(got, denoise_reference(frame[0], 3, *frame[1:], iterations=it, sigma_color=0.7), canonical_nan=True)


@pytest.mark.gpu
def test_gpu_miss_pixels_equal_the_render(gpu_rt, scenes):
    """At a miss pixel the denoised RGBA8 equals render_device's RGBA8 of the same sums."""
    h = gpu_rt.load_world(scenes.default_world())
    W, H = 320, 180
    accum, guides, frame = _gpu_inputs(gpu_rt, h, W, H, 8)
    got, _ = _gpu_denoise(gpu_rt, accum, 8, guides)
    miss = guides["prim"].cpu().numpy() < 0
    render = frame.cpu().numpy().view(np.uint8).reshape(H, W, 4)
    assert miss.any()
    assert np.array_equal(got["pixels"][miss], render[miss])


@pytest.mark.gpu
def test_gpu_each_output_alone_stream_device_and_concurrency(gpu_rt, scenes):
    import torch
    h = gpu_rt.load_world(scenes.c3_world())
    W, H = 320, 180
    accum, guides, _ = _gpu_inputs(gpu_rt, h, W, H, 4)
    arrs = _np((accum, guides, None))
    want = denoise_reference(arrs[0], 4, *arrs[1:])
    gp = [guides[k].data_ptr() for k in ("normal", "position", "albedo", "prim")]

    def outs():
        return (torch.full((H, W, 4), 7, dtype=torch.uint8, device="cuda"),
                torch.full((H, W, 4), 7.0, dtype=torch.float32, device="cuda"))

    # each output alone
    px, col = outs()
    gpu_rt.denoise_device(None, W, H, accum.data_ptr(), 4, *gp, pixels=px.data_ptr())
    assert_same({"pixels": px.cpu().numpy()}, want)
    assert (col == 7).all()
    gpu_rt.denoise_device(None, W, H, accum.data_ptr(), 4, *gp, color=col.data_ptr())
    assert_same({"color": col.cpu().numpy()}, want, canonical_nan=True)
    # a caller's stream, with work ahead of the call on it: the call is ordered after it and returns when written
    s = torch.cuda.Stream()
    px, col = outs()
    torch.cuda.synchronize()
    with torch.cuda.stream(s):
        torch.cuda._sleep(200_000_000)
    gpu_rt.denoise_device(gpu_rt.DenoiseOptions(device=0), W, H, accum.data_ptr(), 4, *gp, px.data_ptr(),
                          col.data_ptr(), stream=s.cuda_stream)
    assert s.query(), "the call returned before its work on the caller's stream was finished"
    assert_same({"pixels": px.cpu().numpy(), "color": col.cpu().numpy()}, want, canonical_nan=True)
    # two calls on two streams, different frames and options: each gives what it gives alone
    other = denoise_reference(arrs[0], 4, *arrs[1:], iterations=2, sigma_color=2.0)
    s2 = torch.cuda.Stream()
    a1, a2 = outs(), outs()
    with torch.cuda.stream(s):
        torch.cuda._sleep(50_000_000)
    with torch.cuda.stream(s2):
        torch.cuda._sleep(50_000_000)
    gpu_rt.denoise_device(None, W, H, accum.data_ptr(), 4, *gp, a1[0].data_ptr(), a1[1].data_ptr(), stream=s.cuda_stream)
    gpu_rt.denoise_device(gpu_rt.DenoiseOptions(iterations=2, sigma_color=2.0), W, H, accum.data_ptr(), 4, *gp,
                          a2[0].data_ptr(), a2[1].data_ptr(), stream=s2.cuda_stream)
    torch.cuda.synchronize()
    assert_same({"pixels": a1[0].cpu().numpy(), "color": a1[1].cpu().numpy()}, want, canonical_nan=True)
    assert_same({"pixels": a2[0].cpu().numpy(), "color": a2[1].cpu().numpy()}, other, canonical_nan=True)
    # `device` names a device other than the current one (with one GPU: the current one, named explicitly); the
    # caller's current device is left as it was
    n = torch.cuda.device_count()
    target = n - 1
    torch.cuda.set_device(0)
    hd = gpu_rt.load_world(scenes.c3_world())
    a_d, g_d, _ = _gpu_inputs(gpu_rt, hd, W, H, 4, device=target)
    arrs_d = _np((a_d, g_d, None))
    px = torch.full((H, W, 4), 7, dtype=torch.uint8, device=f"cuda:{target}")
    gpu_rt.denoise_device(gpu_rt.DenoiseOptions(device=target), W, H, a_d.data_ptr(), 4,
                          *(g_d[k].data_ptr() for k in ("normal", "position", "albedo", "prim")), px.data_ptr())
    assert torch.cuda.current_device() == 0
    assert_same({"pixels": px.cpu().numpy()}, denoise_reference(arrs_d[0], 4, *arrs_d[1:]))
    if n > 1:                                               # a buffer on another device than the options name
        with pytest.raises(gpu_rt.RenderError, match="not device memory of device 0"):
            gpu_rt.denoise_device(gpu_rt.DenoiseOptions(device=0), W, H, a_d.data_ptr(), 4,
                                  *(g_d[k].data_ptr() for k in ("normal", "position", "albedo", "prim")), px.data_ptr())


@pytest.mark.gpu
def test_gpu_zero_options_are_the_defaults(gpu_rt, scenes):
    h = gpu_rt.load_world(scenes.default_world())
    accum, guides, _ = _gpu_inputs(gpu_rt, h, 160, 90, 4)
    a, _ = _gpu_denoise(gpu_rt, accum, 4, guides)
    b, _ = _gpu_denoise(gpu_rt, accum, 4, guides, iterations=gpu_rt.DENOISE_DEFAULT_ITERATIONS,
                        sigma_color=gpu_rt.DENOISE_DEFAULT_SIGMA_COLOR, sigma_normal=gpu_rt.DENOISE_DEFAULT_SIGMA_NORMAL,
                        sigma_plane=gpu_rt.DENOISE_DEFAULT_SIGMA_PLANE)
    assert_same(a, b, canonical_nan=True)


@pytest.mark.gpu
def test_gpu_render_denoised_equals_the_three_calls_and_meets_quality(gpu_rt, scenes):
    """C2's world and camera at 1920x1080, 4 spp: render_denoised is render_device + render_aov + denoise, and its error
    against a 1024-spp frame (linear rgb, hit pixels) is at most half the noisy frame's."""
    W, H = 1920, 1080
    h = gpu_rt.load_world(scenes.default_world())
    got = gpu_rt.render_denoised(h, W, H, gpu_rt.Options(samples_per_pixel=4))
    accum, guides, _ = _gpu_inputs(gpu_rt, h, W, H, 4)
    by_hand = gpu_rt.denoise(accum, 4, guides)
    assert_same({k: v.cpu().numpy() for k, v in got.items()}, {k: v.cpu().numpy() for k, v in by_hand.items()},
                canonical_nan=True)
    ref, _, _ = _gpu_inputs(gpu_rt, h, W, H, 1024)
    prim = guides["prim"].cpu().numpy()
    ref = ref.cpu().numpy() / f32(1024)
    e_noisy = mse_hits(accum.cpu().numpy() / f32(4), ref, prim)
    e_den = mse_hits(got["color"].cpu().numpy(), ref, prim)
    assert e_den <= 0.5 * e_noisy, (e_den, e_noisy)
