"""Variance-guided filtering (rt_svgf_device / svgf / SvgfRenderer): temporal accumulation of the demodulated colour
and its luminance moments, a per-pixel variance estimate, and the a-trous filter with that variance setting each
pixel's colour weight, equal to the numpy reference below bit for bit.

`svgf_reference` restates DESIGN.md §16.1 in numpy float32, vectorised over pixels, with loops over the taps and the
iterations in the kernels' order.  A skipped tap adds +0.0 to sums that start at +0.0 and so are never -0.0, so the
masked sums equal the kernels' branchy ones.  The history lookup and the random frames are test_temporal's.

CPU tests: the boundary (symbols, struct layout, defaults, every rejection), the device header's per-pixel functions
built for the host (tests/svgf_host) against the reference on random and oracle frames, known answers (misses, a
constant colour, a static camera, the colour history) and the quality along a camera path.  GPU tests: the kernels
against the reference on frames the library renders.  Between the GPU and the CPU a NaN is compared as "NaN".
"""
import ctypes as C
import re
import subprocess
from pathlib import Path

import numpy as np
import pytest

import cases
import test_temporal as tt

HERE = Path(__file__).resolve().parent
ROOT = HERE.parent
SVGF_HOST = HERE / "svgf_host"
f32 = np.float32
ALBEDO_FLOOR = f32(2.0 ** -10)                                               # §12.1: a' = max(albedo, 2^-10)
EPS = f32(2.0 ** -20)                                                        # §16.1: il = 1 / (ql g + eps)
DEFAULTS = {"iterations": 5, "max_history": 8, "normal_cos": 0.9, "plane_tol": 0.02, "sigma_luminance": 0.5,
            "sigma_normal": 0.25, "sigma_plane": 0.02}
H5 = {-2: f32(0.0625), -1: f32(0.25), 0: f32(0.375), 1: f32(0.25), 2: f32(0.0625)}   # B3-spline taps
H3 = {-1: f32(0.25), 0: f32(0.5), 1: f32(0.25)}                                       # the variance's Gaussian
OUTPUTS = ("illum", "moments", "length", "color", "pixels")


# ------------------------------------------------------------------------------------------------------- reference

def _dot(a, b):
    return (a[..., 0] * b[..., 0] + a[..., 1] * b[..., 1]) + a[..., 2] * b[..., 2]


def lum(rgb):
    """§16.1: (0.2126 r + 0.7152 g) + 0.0722 b"""
    return (f32(0.2126) * rgb[..., 0] + f32(0.7152) * rgb[..., 1]) + f32(0.0722) * rgb[..., 2]


def _shift(a, dy, dx):
    """(out, inside): out[y, x] = a[y + dy, x + dx] where that lies inside the frame (inside True), else 0."""
    H, W = a.shape[:2]
    out = np.zeros_like(a)
    inside = np.zeros((H, W), bool)
    y0, y1, x0, x1 = max(0, -dy), min(H, H - dy), max(0, -dx), min(W, W - dx)
    if y0 < y1 and x0 < x1:
        out[y0:y1, x0:x1] = a[y0 + dy:y1 + dy, x0 + dx:x1 + dx]
        inside[y0:y1, x0:x1] = True
    return out, inside


def _geometry_u(normal, position, nq, xq, sn, sx):
    """dn_weight's normal and plane terms (u_n, u_x) of tap q for every pixel p."""
    dn = normal - nq
    un = _dot(dn, dn) * sn
    d = _dot(normal, xq - position)
    return un, (d * d) * sx


def _r16(r):
    for _ in range(4):
        r = r * r
    return r


def _opts(o):
    o = {k: (o.get(k) or v) for k, v in DEFAULTS.items()}
    return o


def svgf_reference(accum, spp, position, normal, albedo, prim, camera, prev=None, **options):
    """{"illum", "moments", "length", "color", "pixels", and the stage-2 "variance"} of DESIGN.md §16.1.  prev: None or
    {"camera", "position", "normal", "prim", "illum", "moments", "length"} of the previous frame; a 0 or missing
    option takes its default."""
    o = _opts(options)
    accum, position, normal, albedo = (np.asarray(a, np.float32) for a in (accum, position, normal, albedo))
    prim = np.asarray(prim)
    H, W = prim.shape
    sppf, k = f32(spp), f32(1) / f32(spp)
    sn = f32(1) / ((f32(16) * f32(o["sigma_normal"])) * f32(o["sigma_normal"]))
    sx = f32(1) / ((f32(16) * f32(o["sigma_plane"])) * f32(o["sigma_plane"]))
    ql = (f32(16) * f32(o["sigma_luminance"])) * f32(o["sigma_luminance"])
    hit = prim >= 0
    with np.errstate(all="ignore"):
        # stage 1: demodulation, frame moments, the history of §15.1
        m = accum * k
        ap = np.fmax(albedo, ALBEDO_FLOOR)
        e = m[..., :3] / ap
        l = lum(e)
        l2 = l * l
        illum = np.concatenate([e, l[..., None]], -1)
        mom = np.stack([l, l2], -1)
        length = np.full((H, W), sppf, np.float32)
        if prev is not None:
            cam, pcam = np.asarray(camera, np.float32), np.asarray(prev["camera"], np.float32)
            pprim, pnormal, pposition = (np.asarray(prev[q]) for q in ("prim", "normal", "position"))
            pillum = np.asarray(prev["illum"], np.float32)
            pmom, plength = np.asarray(prev["moments"], np.float32), np.asarray(prev["length"], np.float32)
            ok_p = hit & np.isfinite(position).all(-1) & np.isfinite(normal).all(-1)
            rows, cols = np.mgrid[0:H, 0:W]
            if cam.tobytes() == pcam.tobytes():                              # identity rule
                taps = [(cols, rows, np.ones((H, W), np.float32), ok_p)]
            else:
                x, y, ok = tt.project(pcam, position, W, H)
                ok = ok & ok_p
                x0, y0 = np.floor(x), np.floor(y)
                fx, fy = x - x0, y - y0
                ix = np.where(ok, x0, 0).astype(np.int64)
                iy = np.where(ok, y0, 0).astype(np.int64)
                one = f32(1)
                taps = [(ix, iy, (one - fx) * (one - fy), ok), (ix + 1, iy, fx * (one - fy), ok),
                        (ix, iy + 1, (one - fx) * fy, ok), (ix + 1, iy + 1, fx * fy, ok)]
            sw = np.zeros((H, W), np.float32)
            sc = np.zeros((H, W, 3), np.float32)
            sm = np.zeros((H, W, 2), np.float32)
            sl = np.zeros((H, W), np.float32)
            nc, pt = f32(o["normal_cos"]), f32(o["plane_tol"])
            for qx, qy, wt, ok in taps:                                      # tap order
                inside = ok & (qx >= 0) & (qy >= 0) & (qx < W) & (qy < H) & (wt > 0)
                cx, cy = np.clip(qx, 0, W - 1), np.clip(qy, 0, H - 1)
                acc = inside & (pprim[cy, cx] >= 0)
                acc &= _dot(normal, pnormal[cy, cx]) >= nc
                acc &= np.abs(_dot(normal, pposition[cy, cx] - position)) <= pt
                sw = sw + np.where(acc, wt, f32(0))
                sc = sc + np.where(acc[..., None], wt[..., None] * pillum[cy, cx][..., :3], f32(0))
                sm = sm + np.where(acc[..., None], wt[..., None] * pmom[cy, cx], f32(0))
                sl = sl + np.where(acc, wt * plength[cy, cx], f32(0))
            n = np.fmin(sl / sw, f32(o["max_history"]))                      # fminf: a NaN length gives max_history
            use = (sw >= tt.MIN_WEIGHT) & (n > 0)
            L = n + sppf
            rgb = ((sc / sw[..., None]) * n[..., None] + e * sppf) / L[..., None]
            m1 = ((sm[..., 0] / sw) * n + l * sppf) / L
            m2 = ((sm[..., 1] / sw) * n + l2 * sppf) / L
            illum = np.where(use[..., None], np.concatenate([rgb, lum(rgb)[..., None]], -1), illum)
            mom = np.where(use[..., None], np.stack([m1, m2], -1), mom)
            length = np.where(use, L, length)
        illum = np.where(hit[..., None], illum, m)                           # a miss: m, no moments, spp
        mom = np.where(hit[..., None], mom, f32(0))

        # stage 2: the variance, temporal for L >= 4 spp, else spatial over 7x7 (temporal when no tap is accepted)
        spp4 = f32(4) * sppf
        var_t = np.fmax(mom[..., 1] - mom[..., 0] * mom[..., 0], f32(0))
        sw = np.zeros((H, W), np.float32)
        s1 = np.zeros((H, W), np.float32)
        s2 = np.zeros((H, W), np.float32)
        for dy in range(-3, 4):
            for dx in range(-3, 4):
                hq, inside = _shift(hit, dy, dx)
                un, ux = _geometry_u(normal, position, _shift(normal, dy, dx)[0], _shift(position, dy, dx)[0], sn, sx)
                w = _r16(f32(1) / ((f32(1) + un) * (f32(1) + ux)))
                acc = inside & hq & (w > 0)
                mq = _shift(mom, dy, dx)[0]
                sw = sw + np.where(acc, w, f32(0))
                s1 = s1 + np.where(acc, w * mq[..., 0], f32(0))
                s2 = s2 + np.where(acc, w * mq[..., 1], f32(0))
        mu1 = s1 / sw
        var_s = np.fmax(s2 / sw - mu1 * mu1, f32(0)) * (spp4 / length)
        var = np.where(~(length >= spp4) & (sw > 0), var_s, var_t)
        variance = var

        # stage 3: the a-trous iterations
        ein, out_illum = illum, None
        for it in range(o["iterations"]):
            s = 1 << it
            sk = np.zeros((H, W), np.float32)
            sg = np.zeros((H, W), np.float32)
            for dy in (-1, 0, 1):
                for dx in (-1, 0, 1):
                    hq, inside = _shift(hit, dy, dx)
                    acc = inside & hq
                    kw = H3[dx] * H3[dy]
                    sk = sk + np.where(acc, kw, f32(0))
                    sg = sg + np.where(acc, kw * _shift(var, dy, dx)[0], f32(0))
            il = f32(1) / (ql * (sg / sk) + EPS)
            lp = ein[..., 3]
            sw = np.zeros((H, W), np.float32)
            sc = np.zeros((H, W, 3), np.float32)
            sv = np.zeros((H, W), np.float32)
            for dy in range(-2, 3):
                for dx in range(-2, 3):
                    hq, inside = _shift(hit, dy * s, dx * s)
                    eq = _shift(ein, dy * s, dx * s)[0]
                    lq = eq[..., 3]
                    ul = ((lp - lq) * (lp - lq)) * il
                    un, ux = _geometry_u(normal, position, _shift(normal, dy * s, dx * s)[0],
                                         _shift(position, dy * s, dx * s)[0], sn, sx)
                    w = (H5[dx] * H5[dy]) * _r16(f32(1) / (((f32(1) + ul) * (f32(1) + un)) * (f32(1) + ux)))
                    acc = inside & hq & (w > 0)
                    sw = sw + np.where(acc, w, f32(0))
                    sc = sc + np.where(acc[..., None], w[..., None] * eq[..., :3], f32(0))
                    sv = sv + np.where(acc, (w * w) * _shift(var, dy * s, dx * s)[0], f32(0))
            keep = ~(sw > 0) | ~hit
            rgb = sc / sw[..., None]
            ein = np.where(keep[..., None], ein, np.concatenate([rgb, lum(rgb)[..., None]], -1))
            var = np.where(keep, var, sv / (sw * sw))
            if it == 0:
                out_illum = ein                                              # at a miss: m, from stage 1
        color = np.where(hit[..., None], np.concatenate([ein[..., :3] * ap, m[..., 3:]], -1), m)
    return {"illum": out_illum, "moments": mom, "length": length, "color": color, "pixels": tt.rgba8(color),
            "variance": variance}


def assert_same(got, want, canonical_nan=False, keys=OUTPUTS):
    for key in keys:
        if got.get(key) is None:
            continue
        g, w = np.asarray(got[key]), np.asarray(want[key])
        bad = np.argwhere(tt._bits(g, canonical_nan) != tt._bits(w, canonical_nan))
        assert bad.size == 0, f"{key}: {len(bad)} values differ, first at {bad[0].tolist()}: {g[tuple(bad[0])]} vs {w[tuple(bad[0])]}"


# ----------------------------------------------------------------------------------------------- random frames

def random_frames(seed, W, H, nasty=True):
    """test_temporal's random frames with an albedo (zeros, tiny and NaN values with `nasty`) and a previous frame of
    illum and moments (NaN moments with `nasty`) in place of its colour."""
    (acc, x, n, p, cam), prev = tt.random_frames(seed, W, H, nasty)
    rng = np.random.default_rng(seed + 1)
    albedo = rng.uniform(0.05, 1.0, (H, W, 3)).astype(np.float32)
    mom1 = (rng.random((H, W)) * 2).astype(np.float32)
    moments = np.stack([mom1, mom1 * mom1 + rng.random((H, W)).astype(np.float32)], -1).astype(np.float32)
    if nasty:
        albedo[rng.random((H, W)) < 0.05, 0] = 0.0
        albedo[rng.random((H, W)) < 0.02, 1] = 1e-5
        albedo[rng.random((H, W)) < 0.01, 2] = np.nan
        moments[rng.random((H, W)) < 0.02, 1] = np.nan
        moments[rng.random((H, W)) < 0.02, 0] = -0.5
    illum = prev.pop("color")
    prev.update(illum=illum, moments=moments)
    return (acc, x, n, albedo, p, cam), prev


# ---------------------------------------------------------------------------------------------------------- C ABI

def test_header_declares_the_call_and_the_package_exports_it(rt, tmp_path):
    text = (ROOT / "include" / "raytracer_b200.h").read_text()
    assert "int rt_svgf_device(" in text and "typedef struct RtSvgfOptions" in text
    assert "typedef struct RtSvgfHistory" in text
    assert "rt_svgf_device" in rt.EXPORTED_SYMBOLS and hasattr(rt.lib(), "rt_svgf_device")
    assert rt.lib().rt_abi_version() == 2
    src = tmp_path / "layout.c"
    fields = ["sizeof(RtSvgfOptions)"] + [f"offsetof(RtSvgfOptions, {f})" for f in
                                          ("iterations", "max_history", "normal_cos", "plane_tol", "sigma_luminance",
                                           "sigma_normal", "sigma_plane", "device", "reserved", "stats")] + \
             ["sizeof(RtSvgfHistory)"] + [f"offsetof(RtSvgfHistory, {f})" for f in
                                          ("camera12", "guides", "illum", "moments", "length")]
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "raytracer_b200.h"\n'
                   "int main(void) { printf(\"" + "%zu " * len(fields) + "\\n\", " + ", ".join(fields) +
                   "); return 0; }\n")
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-std=c11", "-I", str(ROOT / "include"), str(src), "-o", str(exe)], check=True)
    got = list(map(int, subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()))
    o, h = rt._SvgfOptions, rt._SvgfHistory
    assert got == [C.sizeof(o)] + [getattr(o, f).offset for f in
                                   ("iterations", "max_history", "normal_cos", "plane_tol", "sigma_luminance",
                                    "sigma_normal", "sigma_plane", "device", "reserved", "stats")] + \
        [C.sizeof(h)] + [getattr(h, f).offset for f in ("camera12", "guides", "illum", "moments", "length")]


def test_defaults_agree_everywhere(rt):
    """The header's RT_SVGF_DEFAULT_*, the host layer's constants, the package's and this reference's."""
    hdr = (ROOT / "include" / "raytracer_b200.h").read_text()
    host = (ROOT / "rust-swift-raytracer_b200" / "csrc" / "rt_host.hpp").read_text()
    for key in DEFAULTS:
        name = key.upper()
        cname = "".join(w.capitalize() for w in key.split("_"))
        h = re.search(r"#define RT_SVGF_DEFAULT_%s ([0-9.]+)[uf]" % name, hdr).group(1)
        c = re.search(r"kSvgfDefault%s\s*=\s*([0-9.]+)[uf];" % cname, host).group(1)
        assert f32(h) == f32(c) == f32(getattr(rt, "SVGF_DEFAULT_" + name)) == f32(DEFAULTS[key]), key


def _host_frame(W=8, H=4):
    (acc, x, n, a, p, cam), prev = random_frames(1, W, H, nasty=False)
    bufs = {"accum": acc, "position": x, "normal": n, "albedo": a, "prim": p,
            "prev_position": prev["position"], "prev_normal": prev["normal"], "prev_prim": prev["prim"],
            "prev_illum": prev["illum"], "prev_moments": prev["moments"], "prev_length": prev["length"],
            "illum": np.full((H, W, 4), 7.0, np.float32), "moments": np.full((H, W, 2), 7.0, np.float32),
            "length": np.full((H, W), 7.0, np.float32), "pixels": np.full((H, W, 4), 7, np.uint8),
            "color": np.full((H, W, 4), 7.0, np.float32)}
    # one arena, buffers back to back in this order on 64-byte boundaries, so that an output placed on or into a
    # buffer overlaps exactly the buffers that follow it here, whatever the heap does
    arena = np.zeros(sum(-(-v.nbytes // 64) * 64 for v in bufs.values()) + 1024, np.uint8)
    off = -arena.ctypes.data % 64
    for k, v in bufs.items():
        view = arena[off:off + v.nbytes].view(v.dtype).reshape(v.shape)
        view[...] = v
        bufs[k] = view
        off += -(-v.nbytes // 64) * 64
    return bufs, cam, prev["camera"]


def _untouched(bufs):
    return all((bufs[k] == 7).all() for k in OUTPUTS)


def _call(rt, bufs, cam, pcam, W=8, H=4, spp=4, opt=None, history=True, **over):
    addr = {k: v.ctypes.data for k, v in bufs.items()}
    addr.update(over)
    hist = {}
    if history:
        hist = dict(prev_camera=over.get("prev_camera_floats", pcam), prev_position=addr["prev_position"],
                    prev_normal=addr["prev_normal"], prev_prim=addr["prev_prim"], prev_illum=addr["prev_illum"],
                    prev_moments=addr["prev_moments"], prev_length=addr["prev_length"])
    rt.svgf_device(opt if opt is not None else rt.SvgfOptions(), W, H, addr["accum"], spp, addr["position"],
                   addr["normal"], addr["albedo"], addr["prim"], over.get("camera_floats", cam), addr["illum"],
                   addr["moments"], addr["length"], addr["pixels"], addr["color"], **hist)


REJECTED = [
    ("iterations", dict(opt=dict(iterations=11)), "iterations must be in 1..10"),
    ("max_history", dict(opt=dict(max_history=2 ** 20 + 1)), "max_history must be in 1..2^20 (0: the default, 8)"),
    ("normal_cos_big", dict(opt=dict(normal_cos=-1.5)), "normal_cos must be finite and in [-1, 1]"),
    ("normal_cos_nan", dict(opt=dict(normal_cos=float("nan"))), "normal_cos must be finite and in [-1, 1]"),
    ("plane_tol_negative", dict(opt=dict(plane_tol=-0.1)), "plane_tol must be finite and > 0"),
    ("plane_tol_inf", dict(opt=dict(plane_tol=float("inf"))), "plane_tol must be finite and > 0"),
    ("sigma_luminance_negative", dict(opt=dict(sigma_luminance=-1.0)), "sigma_luminance must be finite and > 0"),
    ("sigma_luminance_nan", dict(opt=dict(sigma_luminance=float("nan"))), "sigma_luminance must be finite and > 0"),
    ("sigma_luminance_inf", dict(opt=dict(sigma_luminance=float("inf"))), "sigma_luminance must be finite and > 0"),
    ("sigma_normal_nan", dict(opt=dict(sigma_normal=float("nan"))), "sigma_normal must be finite and > 0"),
    ("sigma_plane_inf", dict(opt=dict(sigma_plane=float("inf"))), "sigma_plane must be finite and > 0"),
    ("spp_zero", dict(spp=0), "spp must be >= 1"),
    ("accum_null", dict(over=dict(accum=0)), "the accum buffer is NULL"),
    ("position_null", dict(over=dict(position=0)), "the position buffer is NULL"),
    ("normal_null", dict(over=dict(normal=0)), "the normal buffer is NULL"),
    ("albedo_null", dict(over=dict(albedo=0)), "the albedo buffer is NULL"),
    ("prim_null", dict(over=dict(prim=0)), "the prim buffer is NULL"),
    ("camera_null", dict(camera=None), "the camera is NULL"),
    ("camera_inf", dict(camera=tt.BAD_CAM), "the camera has a non-finite float"),
    ("prev_camera_null", dict(pcam=None), "only partly given: its camera is NULL"),
    ("prev_camera_nan", dict(pcam=np.where(np.arange(12) == 4, np.nan, 1.0).astype(np.float32)),
     "the previous camera has a non-finite float"),
    ("prev_normal_null", dict(over=dict(prev_normal=0)), "only partly given: the previous normal is NULL"),
    ("prev_illum_null", dict(over=dict(prev_illum=0)), "only partly given: the previous illum is NULL"),
    ("prev_moments_null", dict(over=dict(prev_moments=0)), "only partly given: the previous moments is NULL"),
    ("prev_length_null", dict(over=dict(prev_length=0)), "only partly given: the previous length is NULL"),
    ("illum_null", dict(over=dict(illum=0)), "the illum output is NULL"),
    ("moments_null", dict(over=dict(moments=0)), "the moments output is NULL"),
    ("length_null", dict(over=dict(length=0)), "the length output is NULL"),
    ("pixels_and_color_null", dict(over=dict(pixels=0, color=0)), "both outputs (pixels, color) are NULL"),
    ("width_zero", dict(W=0), "at least 1x1"),
    ("too_tall", dict(H=2 ** 30), "framebuffer too large"),
    ("illum_over_prev_illum", dict(over="illum:prev_illum"), "the illum output overlaps the previous illum input"),
    ("moments_over_prev_moments", dict(over="moments:prev_moments"),
     "the moments output overlaps the previous moments input"),
    ("length_over_prev_length", dict(over="length:prev_length"), "the length output overlaps the previous length input"),
    ("accum_misaligned", dict(over="accum:accum@4"), "the accum buffer is not 16-byte aligned"),
    ("prev_illum_misaligned", dict(over="prev_illum:prev_illum@8"), "the previous illum buffer is not 16-byte aligned"),
    ("prev_moments_misaligned", dict(over="prev_moments:prev_moments@4"),
     "the previous moments buffer is not 8-byte aligned"),
    ("illum_misaligned", dict(over="illum:illum@4"), "the illum buffer is not 16-byte aligned"),
    ("moments_misaligned", dict(over="moments:moments@4"), "the moments buffer is not 8-byte aligned"),
    ("color_misaligned", dict(over="color:color@12"), "the color buffer is not 16-byte aligned"),
    ("color_over_albedo_tail", dict(over="color:albedo+"), "the color output overlaps the albedo input"),
    ("moments_over_illum", dict(over="moments:illum"), "the moments output overlaps the illum output"),
    ("pixels_over_length", dict(over="pixels:length"), "the pixels output overlaps the length output"),
    ("color_over_pixels", dict(over="color:pixels"), "the color output overlaps the pixels output"),
]


@pytest.mark.parametrize("name,spec,text", REJECTED, ids=[r[0] for r in REJECTED])
def test_rejections_fail_on_the_host(rt, name, spec, text):
    bufs, cam, pcam = _host_frame()
    over = spec.get("over", {})
    if isinstance(over, str):                               # "out:in": the output placed on (or into) another buffer
        out, inp = over.split(":")                          # "in+": its last 16 bytes, "in@k": k bytes in
        inp, _, shift = inp.partition("@")
        tail = inp.endswith("+")
        inp = inp.rstrip("+")
        over = {out: bufs[inp].ctypes.data + (bufs[inp].nbytes - 16 if tail else int(shift or 0))}
    over = dict(over)
    if "camera" in spec:
        over["camera_floats"] = spec["camera"]
    if "pcam" in spec:
        over["prev_camera_floats"] = spec["pcam"]
    with pytest.raises(rt.RenderError) as e:
        _call(rt, bufs, cam, pcam, W=spec.get("W", 8), H=spec.get("H", 4), spp=spec.get("spp", 4),
              opt=rt.SvgfOptions(**spec.get("opt", {})), **over)
    assert str(e.value).startswith("svgf: ") and text in str(e.value), str(e.value)
    assert _untouched(bufs)


def test_null_options_struct_sizes_guides_and_history_members(rt):
    L = rt.lib()
    bufs, cam, pcam = _host_frame()
    g = rt.AovBuffers(C.sizeof(rt.AovBuffers), 0, None, bufs["position"].ctypes.data, bufs["normal"].ctypes.data,
                      bufs["albedo"].ctypes.data, bufs["prim"].ctypes.data)
    c12 = (C.c_float * 12)(*cam)
    args = (8, 4, bufs["accum"].ctypes.data, 4)
    outs = tuple(bufs[k].ctypes.data for k in ("illum", "moments", "length", "pixels", "color")) + (None,)
    assert L.rt_svgf_device(None, *args, C.byref(g), c12, None, *outs) != 0
    assert "rt_svgf_device: options is NULL" in rt.last_error()
    o = rt.SvgfOptions()._c(None)
    o.struct_size = 40
    assert L.rt_svgf_device(C.byref(o), *args, C.byref(g), c12, None, *outs) != 0
    assert "options->struct_size" in rt.last_error()
    o = rt.SvgfOptions()._c(None)
    assert L.rt_svgf_device(C.byref(o), *args, None, c12, None, *outs) != 0
    assert "guides is NULL" in rt.last_error()
    pc = (C.c_float * 12)(*pcam)
    pg = rt.AovBuffers(C.sizeof(rt.AovBuffers), 0, None, bufs["prev_position"].ctypes.data,
                       bufs["prev_normal"].ctypes.data, None, bufs["prev_prim"].ctypes.data)
    h = rt._SvgfHistory(C.sizeof(rt._SvgfHistory) - 8, 0, C.cast(pc, C.POINTER(C.c_float)), C.pointer(pg),
                        bufs["prev_illum"].ctypes.data, bufs["prev_moments"].ctypes.data,
                        bufs["prev_length"].ctypes.data)
    assert L.rt_svgf_device(C.byref(o), *args, C.byref(g), c12, C.byref(h), *outs) != 0
    assert "history->struct_size" in rt.last_error()
    h.struct_size = C.sizeof(rt._SvgfHistory)
    h.guides = None                                          # a history without its guides is only partly given
    assert L.rt_svgf_device(C.byref(o), *args, C.byref(g), c12, C.byref(h), *outs) != 0
    assert "svgf: the previous frame is only partly given: the previous position is NULL" in rt.last_error()
    empty = rt._SvgfHistory(C.sizeof(rt._SvgfHistory), 0, None, None, None, None, None)
    assert L.rt_svgf_device(C.byref(o), *args, C.byref(g), c12, C.byref(empty), *outs) != 0
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
    subprocess.run(["make", "-C", str(SVGF_HOST), "build/libsvgf_hostsim.so"], check=True, capture_output=True)
    L = C.CDLL(str(SVGF_HOST / "build" / "libsvgf_hostsim.so"))
    L.hostsim_svgf.restype = C.c_int
    L.hostsim_svgf.argtypes = [C.c_uint32, C.c_uint32, C.c_void_p, C.c_int32] + [C.c_void_p] * 12 + \
                              [C.c_uint32, C.c_uint32] + [C.c_float] * 5 + [C.c_void_p] * 5
    return L


def hostsim_svgf(L, accum, spp, position, normal, albedo, prim, camera, prev=None, **options):
    o = _opts(options)
    H, W = prim.shape
    keep = []

    def a(x, dt=np.float32):
        if x is None:
            return None
        x = np.ascontiguousarray(x, dt)
        keep.append(x)
        return x.ctypes.data

    p = prev or {}
    out = {"illum": np.zeros((H, W, 4), np.float32), "moments": np.zeros((H, W, 2), np.float32),
           "length": np.zeros((H, W), np.float32), "color": np.zeros((H, W, 4), np.float32),
           "pixels": np.zeros((H, W, 4), np.uint8)}
    rc = L.hostsim_svgf(W, H, a(accum), spp, a(position), a(normal), a(albedo), a(prim, np.int32), a(camera),
                        a(p.get("camera")), a(p.get("position")), a(p.get("normal")), a(p.get("prim"), np.int32),
                        a(p.get("illum")), a(p.get("moments")), a(p.get("length")), int(o["iterations"]),
                        int(o["max_history"]), float(o["normal_cos"]), float(o["plane_tol"]),
                        float(o["sigma_luminance"]), float(o["sigma_normal"]), float(o["sigma_plane"]),
                        *(out[k].ctypes.data for k in OUTPUTS))
    assert rc == 0
    return out


@pytest.mark.parametrize("W,H", [(1, 1), (7, 1), (1, 5), (123, 77)])
@pytest.mark.parametrize("iterations", [1, 5, 10])
def test_device_functions_on_host_equal_reference_on_random_frames(hostsim, W, H, iterations):
    young = old = 0
    for seed in range(3):
        (acc, x, n, al, p, cam), prev = random_frames(100 * seed + W + H + iterations, W, H)
        spp = (1, 4, 9)[seed]
        opts = dict(iterations=iterations, max_history=(0, 5, 1000)[seed], normal_cos=(0.0, 0.5, -1.0)[seed],
                    plane_tol=(0.0, 0.05, 0.5)[seed], sigma_luminance=(0.0, 1.0, 16.0)[seed],
                    sigma_normal=(0.0, 0.5, 0.1)[seed], sigma_plane=(0.0, 0.1, 0.01)[seed])
        for pv in (None, prev, dict(prev, camera=cam)):                    # no history, reprojection, identity rule
            want = svgf_reference(acc, spp, x, n, al, p, cam, pv, **opts)
            assert_same(hostsim_svgf(hostsim, acc, spp, x, n, al, p, cam, pv, **opts), want)
            hit = p >= 0
            young += int(np.sum(hit & (want["length"] < 4 * spp)))
            old += int(np.sum(hit & (want["length"] >= 4 * spp)))
    if W * H > 1000:                                                       # both sides of L = 4 spp
        assert young > 0 and old > 0


def _svgf_path(frames, spp, sim=None, **opts):
    """svgf_reference (and the host build when `sim` is given) along oracle frames; returns the outputs."""
    results, prev = [], None
    for accum, g, cam in frames:
        args = (accum, spp, g["position"], g["normal"], g["albedo"], g["prim"], cam, prev)
        out = svgf_reference(*args, **opts)
        if sim is not None:
            assert_same(hostsim_svgf(sim, *args, **opts), out)
        results.append(out)
        prev = {"camera": cam, "position": g["position"], "normal": g["normal"], "prim": g["prim"],
                "illum": out["illum"], "moments": out["moments"], "length": out["length"]}
    return results


@pytest.mark.parametrize("key,camera,W,H,spp", [("default", "file", 160, 90, 4), ("example", "file", 123, 77, 3),
                                                ("c3", "file", 96, 54, 2)])
def test_device_functions_on_host_equal_reference_on_oracle_frames(hostsim, ob, scenes, key, camera, W, H, spp):
    frames, _, _ = tt._oracle_frames(ob, scenes, key, camera, W, H, spp, 3)
    frames = frames + [frames[-1]]                                         # and a static frame
    _svgf_path(frames, spp, hostsim)
    outs = _svgf_path(frames, spp, hostsim, max_history=64)                # both sides of L = 4 spp
    hit = frames[-1][1]["prim"] >= 0
    assert (outs[-1]["length"][hit] >= 4 * spp).any() and (outs[-1]["length"][hit] < 4 * spp).any()
    _svgf_path(frames, spp, hostsim, iterations=2, max_history=4, normal_cos=0.5, plane_tol=0.1,
               sigma_luminance=1.0, sigma_normal=0.5, sigma_plane=0.05)


# ------------------------------------------------------------------------------------------------ known answers

def test_misses_are_the_mean_and_the_oracle_rgba8(ob, scenes):
    W, H, spp = 123, 77, 3
    cam, world = cases.oracle_scene(ob, scenes, "example", "file")
    pixels, _, accum = ob.ray_trace(world, cam, W, H, spp, 8, want_accum=True)
    import test_aov
    g = test_aov.primary_hits(ob, world, cam, W, H, fixed_jitter=True)
    out = svgf_reference(accum, spp, g["position"], g["normal"], g["albedo"], g["prim"], cam.floats())
    miss = g["prim"] < 0
    assert 0 < miss.mean() < 1
    m = accum * (f32(1) / f32(spp))
    for key in ("color", "illum"):
        assert (tt._bits(out[key][miss]) == tt._bits(m[miss])).all()
    assert np.array_equal(out["pixels"][miss], pixels[miss])
    assert (out["moments"][miss] == 0).all() and (out["length"] == f32(spp)).all()


def test_constant_colour_passes_unchanged():
    """Every hit pixel of one demodulated colour, seen from two cameras: the variance is 0 up to the rounding of
    mu2 - mu1^2 (at most 32 ulp of l^2, where that difference cancels), and the filter returns the colour within 4
    ulp, the rounding of a weighted mean of up to 25 rounded products (3 ulp after one iteration, 4 after five)."""
    W, H, spp = 48, 32, 2
    (acc, x, n, al, p, cam), prev = random_frames(5, W, H, nasty=False)
    e = np.float32([0.3, 0.55, 0.8])
    al = (f32(2) ** -np.random.default_rng(6).integers(0, 4, (H, W, 3))).astype(np.float32)   # e * a' * spp is exact
    acc = np.concatenate([(e * al) * f32(spp), np.full((H, W, 1), 3.0, np.float32)], -1).astype(np.float32)
    p[:, :5] = -1
    hit = p >= 0
    first = svgf_reference(acc, spp, x, n, al, p, cam)
    ed = (acc[..., :3] * (f32(1) / f32(spp))) / np.fmax(al, ALBEDO_FLOOR)   # the colour as the kernel demodulates it
    prev = dict(prev, illum=first["illum"], moments=first["moments"], length=first["length"])
    for out in (first, svgf_reference(acc, spp, x, n, al, p, cam, prev)):
        assert (out["variance"][hit] <= f32(32) * np.finfo(np.float32).eps * (lum(e) * lum(e))).all()
        assert (out["variance"][hit] == 0).mean() > 0.5
        ulp = np.abs(np.ascontiguousarray(out["illum"][..., :3]).view(np.int32).astype(np.int64) -
                     ed.view(np.int32).astype(np.int64))
        assert ulp[hit].max() <= 4, ulp[hit].max()
        got = np.ascontiguousarray(out["color"][..., :3] / np.fmax(al, ALBEDO_FLOOR))   # a' is a power of 2
        ulp = np.abs(got.view(np.int32).astype(np.int64) - ed.view(np.int32).astype(np.int64))
        assert ulp[hit].max() <= 4, ulp[hit].max()


def test_static_camera_accumulates_the_moments(ob, scenes):
    """k frames of n spp with a static camera and max_history above k*n: at hit pixels length k*n exactly, and the
    moments the running means of the frames' own (l, l*l) within a relative 1e-5."""
    W, H, n, k = 96, 54, 4, 5
    frames, _, _ = tt._oracle_frames(ob, scenes, "default", "file", W, H, n, k, static=True)
    last = _svgf_path(frames, n, max_history=1000)[-1]
    ls = []
    for accum, g, _ in frames:
        e = (accum[..., :3] * (f32(1) / f32(n))) / np.fmax(g["albedo"], ALBEDO_FLOOR)
        ls.append(lum(e).astype(np.float64))
    ls = np.stack(ls)
    hit = frames[-1][1]["prim"] >= 0
    assert hit.mean() > 0.5
    assert (last["length"][hit] == f32(n * k)).all()
    assert np.allclose(last["moments"][..., 0][hit], ls.mean(0)[hit], rtol=1e-5, atol=0)
    assert np.allclose(last["moments"][..., 1][hit], (ls * ls).mean(0)[hit], rtol=1e-5, atol=0)


def test_illum_is_the_first_iteration(hostsim, ob, scenes):
    """illum_out is iteration 0's output: the same for 5 iterations and for 1, where the colour is illum * a'."""
    W, H, spp = 96, 54, 2
    frames, _, _ = tt._oracle_frames(ob, scenes, "c3", "file", W, H, spp, 2)
    prev = None
    for accum, g, cam in frames:
        args = (accum, spp, g["position"], g["normal"], g["albedo"], g["prim"], cam, prev)
        five, one = hostsim_svgf(hostsim, *args), hostsim_svgf(hostsim, *args, iterations=1)
        assert_same(one, svgf_reference(*args, iterations=1))
        assert (tt._bits(five["illum"]) == tt._bits(one["illum"])).all()
        hit = g["prim"] >= 0
        assert (tt._bits(one["color"][..., :3][hit]) ==
                tt._bits((one["illum"][..., :3] * np.fmax(g["albedo"], ALBEDO_FLOOR))[hit])).all()
        assert not np.array_equal(five["color"], one["color"])
        prev = {"camera": cam, "position": g["position"], "normal": g["normal"], "prim": g["prim"],
                "illum": five["illum"], "moments": five["moments"], "length": five["length"]}


def test_quality_along_a_camera_path(ob, scenes):
    """world.txt at 160x90, 8 frames of 4 spp along §15.4's camera path, against 1024 spp of each frame's camera: at
    every frame 1..7 the error is at most half the noisy 4-spp frame's, and at the last frame at most temporal
    accumulation's (DESIGN.md §16.4 records the ratios)."""
    W, H, spp = 160, 90, 4
    frames, world, cams = tt._oracle_frames(ob, scenes, "default", "file", W, H, spp, 8)
    outs = _svgf_path(frames, spp)
    temporal = tt._run_path(frames, spp)
    for i in range(1, len(frames)):
        _, _, ref = ob.ray_trace(world, cams[i], W, H, 1024, 8, want_accum=True, sample_begin=10_000)
        ref = ref / f32(1024)
        prim = frames[i][1]["prim"]
        e_noisy = tt.mse_hits(frames[i][0] / f32(spp), ref, prim)
        e_svgf = tt.mse_hits(outs[i]["color"], ref, prim)
        assert e_svgf <= 0.5 * e_noisy, (i, e_svgf, e_noisy)
        if i == len(frames) - 1:
            e_temporal = tt.mse_hits(temporal[i]["color"], ref, prim)
            assert e_svgf <= e_temporal, (e_svgf, e_temporal)


# ------------------------------------------------------------------------------------------------------------ GPU

def _gpu_frame(gpu_rt, h, W, H, spp, depth=8, sample_begin=0, device=0):
    """test_temporal's frame: accum, render_aov's guides at pixel centres, the RGBA8 frame, the camera floats."""
    return tt._gpu_frame(gpu_rt, h, W, H, spp, depth, sample_begin, device)


def _np_guides(g):
    return {k: g[k].cpu().numpy() for k in ("position", "normal", "albedo", "prim")}


def _np_prev(cam, g, out):
    return {"camera": cam, "position": g["position"], "normal": g["normal"], "prim": g["prim"],
            "illum": out["illum"], "moments": out["moments"], "length": out["length"]}


def _gpu_path_against_reference(gpu_rt, h, W, H, spp, depth=8, frames=3, **opts):
    """Frames along a camera path (then one more with the camera standing still), each filtered on the GPU from the
    GPU's own previous outputs, against the reference of the same inputs."""
    prev_t, prev_np = None, None
    for i in range(frames + 1):
        if 0 < i < frames:
            gpu_rt.move_camera_position(h, *tt.PATH_STEP)
        accum, g, _, cam = _gpu_frame(gpu_rt, h, W, H, spp, depth, sample_begin=spp * i)
        st = gpu_rt.RenderStats()
        out = gpu_rt.svgf(accum, spp, g, cam, prev_t, gpu_rt.SvgfOptions(**opts), stats=st)
        got = {k: v.cpu().numpy() for k, v in out.items()}
        gn = _np_guides(g)
        want = svgf_reference(accum.cpu().numpy(), spp, gn["position"], gn["normal"], gn["albedo"], gn["prim"], cam,
                              prev_np, **opts)
        assert_same(got, want, canonical_nan=True)
        iterations = opts.get("iterations") or DEFAULTS["iterations"]
        assert st.launches == 2 + iterations and st.rays == 0 and st.samples == 0 and st.kernel_ms > 0
        assert st.total_ms >= st.kernel_ms and st.block == 256 and st.grid == ((W + 31) // 32) * ((H + 7) // 8)
        prev_t = {"camera": cam, "guides": g, "illum": out["illum"], "moments": out["moments"], "length": out["length"]}
        prev_np = _np_prev(cam, gn, got)


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
    _gpu_path_against_reference(gpu_rt, h, 320, 180, 2, frames=2, iterations=10, max_history=3, normal_cos=0.5,
                                plane_tol=0.1, sigma_luminance=1.5, sigma_normal=0.5, sigma_plane=0.05)


@pytest.mark.gpu
def test_gpu_random_frames_with_nans(gpu_rt):
    import torch
    (acc, x, n, al, p, cam), prev = random_frames(77, 123, 77)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()   # noqa: E731
    guides = {"position": t(x), "normal": t(n), "albedo": t(al), "prim": t(p)}
    pg = {"position": t(prev["position"]), "normal": t(prev["normal"]), "prim": t(prev["prim"])}
    for pv in (None, prev, dict(prev, camera=cam)):
        prev_t = None if pv is None else {"camera": pv["camera"], "guides": pg, "illum": t(prev["illum"]),
                                          "moments": t(prev["moments"]), "length": t(prev["length"])}
        got = gpu_rt.svgf(t(acc), 3, guides, cam, prev_t, gpu_rt.SvgfOptions(plane_tol=0.05, iterations=3))
        want = svgf_reference(acc, 3, x, n, al, p, cam, pv, plane_tol=0.05, iterations=3)
        assert_same({k: v.cpu().numpy() for k, v in got.items()}, want, canonical_nan=True)


@pytest.mark.gpu
def test_gpu_miss_pixels_equal_the_render(gpu_rt, scenes):
    h = gpu_rt.load_world(scenes.default_world())
    W, H = 320, 180
    accum, g, frame, cam = _gpu_frame(gpu_rt, h, W, H, 8)
    out = gpu_rt.svgf(accum, 8, g, cam)
    miss = g["prim"].cpu().numpy() < 0
    assert miss.any()
    assert np.array_equal(out["pixels"].cpu().numpy()[miss], frame.cpu().numpy().view(np.uint8).reshape(H, W, 4)[miss])


@pytest.mark.gpu
def test_gpu_svgf_renderer(gpu_rt, scenes):
    """A static camera keeps adding samples (length k*n at hits, with max_history above it); a camera move keeps part
    of the history; reset() and a resize drop all of it.  Each frame equals svgf() of its own inputs."""
    W, H, n, k = 320, 180, 4, 4
    h = gpu_rt.load_world(scenes.default_world())
    r = gpu_rt.SvgfRenderer(W, H, gpu_rt.Options(samples_per_pixel=n), gpu_rt.SvgfOptions(max_history=1000))
    for _ in range(k):
        out = r.frame(h)
    hit = r._prev["guides"]["prim"].cpu().numpy() >= 0
    assert (out["length"].cpu().numpy()[hit] == n * k).all()
    assert (out["length"].cpu().numpy()[~hit] == n).all()
    gpu_rt.move_camera_position(h, *tt.PATH_STEP)
    moved = r.frame(h)["length"].cpu().numpy()
    assert (moved > n).mean() > 0.5 and (moved == n).any()
    r.reset()
    assert (r.frame(h)["length"] == n).all()
    assert (r.frame(h)["length"] > n).any()
    r.width, r.height = 160, 90
    out = r.frame(h)
    assert (out["length"] == n).all() and tuple(out["pixels"].shape) == (90, 160, 4)


@pytest.mark.gpu
def test_gpu_outputs_streams_device_and_stats(gpu_rt, scenes):
    import torch
    h = gpu_rt.load_world(scenes.c3_world())
    W, H = 320, 180
    a0, g0, _, c0 = _gpu_frame(gpu_rt, h, W, H, 4)
    gpu_rt.move_camera_position(h, *tt.PATH_STEP)
    a1, g1, _, c1 = _gpu_frame(gpu_rt, h, W, H, 4, sample_begin=4)
    n0, n1 = _np_guides(g0), _np_guides(g1)
    want0 = svgf_reference(a0.cpu().numpy(), 4, n0["position"], n0["normal"], n0["albedo"], n0["prim"], c0)
    want1 = svgf_reference(a1.cpu().numpy(), 4, n1["position"], n1["normal"], n1["albedo"], n1["prim"], c1,
                           _np_prev(c0, n0, want0))
    ptr = lambda g: tuple(g[k].data_ptr() for k in ("position", "normal", "albedo", "prim"))   # noqa: E731

    def outs(device="cuda"):                             # filled before the library's stream writes them
        o = {"illum": torch.full((H, W, 4), 7.0, device=device), "moments": torch.full((H, W, 2), 7.0, device=device),
             "length": torch.full((H, W), 7.0, device=device),
             "pixels": torch.full((H, W, 4), 7, dtype=torch.uint8, device=device),
             "color": torch.full((H, W, 4), 7.0, device=device)}
        torch.cuda.synchronize()
        return o

    def np_(o):
        return {k: v.cpu().numpy() for k, v in o.items()}

    def run(o, a, g, c, opts=None, stream=0, stats=None, hist=None):
        gpu_rt.svgf_device(opts, W, H, a.data_ptr(), 4, *ptr(g), c, o["illum"].data_ptr(), o["moments"].data_ptr(),
                           o["length"].data_ptr(), o["pixels"].data_ptr() if "pixels" in o else 0,
                           o["color"].data_ptr() if "color" in o else 0, stream=stream, stats=stats, **(hist or {}))

    # each optional output alone
    for alone in ("pixels", "color"):
        o = outs()
        other = o.pop("color" if alone == "pixels" else "pixels")
        run(o, a0, g0, c0)
        assert_same(np_(o), want0, canonical_nan=True, keys=("illum", "moments", "length", alone))
        assert (other == 7).all()
    # a chained pair on a caller's stream behind a busy kernel: the scratch makes each call wait for its own work
    s = torch.cuda.Stream()
    oa, ob_ = outs(), outs()
    with torch.cuda.stream(s):
        torch.cuda._sleep(100_000_000)
    run(oa, a0, g0, c0, opts=gpu_rt.SvgfOptions(device=0), stream=s.cuda_stream)
    assert s.query(), "the call returned before its work on the caller's stream was finished"
    hist = dict(prev_camera=c0, prev_position=g0["position"].data_ptr(), prev_normal=g0["normal"].data_ptr(),
                prev_prim=g0["prim"].data_ptr(), prev_illum=oa["illum"].data_ptr(),
                prev_moments=oa["moments"].data_ptr(), prev_length=oa["length"].data_ptr())
    run(ob_, a1, g1, c1, stream=s.cuda_stream, hist=hist)
    assert_same(np_(oa), want0, canonical_nan=True)
    assert_same(np_(ob_), want1, canonical_nan=True)
    # two calls on two streams share the device's scratch: each is finished before the next one starts
    s2 = torch.cuda.Stream()
    oc, od = outs(), outs()
    with torch.cuda.stream(s2):
        torch.cuda._sleep(100_000_000)
    run(oc, a1, g1, c1, stream=s2.cuda_stream, hist=hist)
    run(od, a0, g0, c0, stream=s.cuda_stream)
    assert_same(np_(oc), want1, canonical_nan=True)
    assert_same(np_(od), want0, canonical_nan=True)
    # stats
    st = gpu_rt.RenderStats()
    run(outs(), a0, g0, c0, opts=gpu_rt.SvgfOptions(iterations=3), stats=st)
    assert st.kernel_ms > 0 and st.launches == 5 and st.block == 256 and st.rays == 0 and st.samples == 0
    assert st.grid == ((W + 31) // 32) * ((H + 7) // 8) and st.total_ms >= st.kernel_ms
    # `device` names a device explicitly (the last one); the caller's current device is left as it was
    target = torch.cuda.device_count() - 1
    torch.cuda.set_device(0)
    hd = gpu_rt.load_world(scenes.c3_world())
    a_d, g_d, _, c_d = _gpu_frame(gpu_rt, hd, W, H, 4, device=target)
    o = outs(f"cuda:{target}")
    torch.cuda.synchronize(target)
    run(o, a_d, g_d, c_d, opts=gpu_rt.SvgfOptions(device=target))
    assert torch.cuda.current_device() == 0
    nd = _np_guides(g_d)
    assert_same(np_(o), svgf_reference(a_d.cpu().numpy(), 4, nd["position"], nd["normal"], nd["albedo"], nd["prim"],
                                       c_d), canonical_nan=True)
