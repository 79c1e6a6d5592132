"""Variance-guided filtering against the temporal + denoise chain: timing, quality along a camera path, and the sweep
that chose its defaults, on one GPU.

    python scripts/svgf_bench.py [--reps 20] [--out DIR]

Timing: for the default world (C2's world and camera) and C3, at 1920x1080 and 3840x2160, on a frame whose camera
moved since the previous one (the reprojection path), the kernel time (RenderStats.kernel_ms: CUDA events around all
launches of a call) of rt_svgf_device with default options, alternated with the chain it replaces:
rt_temporal_accumulate_device followed by rt_denoise_device of its colour (spp 1), both with default options.  --reps
repetitions each, with the L2 flushed (256 MiB write) before each call; median, min and max, with the card's name and
power limit read in the same run.

Quality: along a path of 8 frames of 4 spp (the camera moved by move_camera_position between frames) at 1920x1080,
the mean squared error (linear rgb, hit pixels) of each frame's filtered colour, for SVGF and for the chain, and of
its own 4-spp mean, all against a 1024-spp frame of that frame's camera (a disjoint sample range); the ratio per frame.

Sweep: the per-frame ratios for sigma_luminance x max_history on both worlds.
Prints one JSON line; --out DIR also writes it to DIR/svgf_bench.json.
"""
from __future__ import annotations

import argparse
import importlib
import itertools
import json
import statistics
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

STEP = (0.04, 0.0, 0.02)                  # camera move per frame, as tests/test_temporal.py's path
FRAMES = 8
SWEEP_SIGMA_LUMINANCE = (0.5, 1.0, 2.0, 4.0, 8.0)
SWEEP_MAX_HISTORY = (8, 16, 32, 64)


def card() -> str:
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--worlds", default="default,c3")
    ap.add_argument("--sizes", default="1920x1080,3840x2160")
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    import torch
    rt = importlib.import_module("rust-swift-raytracer_b200")
    scenes = importlib.import_module("rust-swift-raytracer_b200.scenes")
    if rt.device_count() < 1:
        raise SystemExit("svgf_bench needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)        # > 126 MB L2

    def frame(h, W, H, spp, sample_begin=0):
        accum = torch.empty((H, W, 4), dtype=torch.float32, device=dev)
        px = torch.empty((H, W), dtype=torch.int32, device=dev)
        rt.render_device(h, rt.Options(samples_per_pixel=spp, accum_out=True, sample_begin=sample_begin, device=0),
                         W, H, px.data_ptr(), accum.data_ptr())
        torch.cuda.synchronize()
        return accum

    def guides(h, W, H):
        return rt.render_aov(h, W, H, rt.Options(fixed_jitter=True, device=0))

    def mse(color, ref, hit):
        d = (color[..., :3].double() - ref[..., :3].double())[hit]
        return float((d * d).mean())

    def ptrs(g, *keys):
        return [g[k].data_ptr() for k in keys]

    result = {"card": card(), "reps": a.reps, "l2": "flushed before each call (256 MiB write)",
              "defaults": {k.lower(): getattr(rt, "SVGF_DEFAULT_" + k) for k in
                           ("ITERATIONS", "MAX_HISTORY", "NORMAL_COS", "PLANE_TOL", "SIGMA_LUMINANCE", "SIGMA_NORMAL",
                            "SIGMA_PLANE")},
              "path": {"frames": FRAMES, "spp": 4, "step": STEP}, "timing": {}, "quality": {}, "sweep": {}}
    for key in a.worlds.split(","):
        text = getattr(scenes, key + "_world")()
        for size in a.sizes.split(","):
            W, H = map(int, size.split("x"))
            h = rt.load_world(text)
            a0, g0, c0 = frame(h, W, H, 1), guides(h, W, H), h.camera_floats()
            sv0 = rt.svgf(a0, 1, g0, c0)
            tp0 = rt.temporal_accumulate(a0, 1, g0, c0, pixels=False)
            rt.move_camera_position(h, *STEP)
            a1, g1, c1 = frame(h, W, H, 1, 1), guides(h, W, H), h.camera_floats()
            f4 = lambda: torch.empty((H, W, 4), dtype=torch.float32, device=dev)   # noqa: E731
            ill, col, tcol, dcol = f4(), f4(), f4(), f4()
            mom = torch.empty((H, W, 2), dtype=torch.float32, device=dev)
            ln, tln = (torch.empty((H, W), dtype=torch.float32, device=dev) for _ in range(2))
            pix, dpix = (torch.empty((H, W, 4), dtype=torch.uint8, device=dev) for _ in range(2))
            pos, nrm, alb, prm = ptrs(g1, "position", "normal", "albedo", "prim")
            pg = dict(prev_camera=c0, prev_position=g0["position"].data_ptr(), prev_normal=g0["normal"].data_ptr(),
                      prev_prim=g0["prim"].data_ptr())

            def call_svgf(st):
                rt.svgf_device(None, W, H, a1.data_ptr(), 1, pos, nrm, alb, prm, c1, ill.data_ptr(), mom.data_ptr(),
                               ln.data_ptr(), pix.data_ptr(), col.data_ptr(), prev_illum=sv0["illum"].data_ptr(),
                               prev_moments=sv0["moments"].data_ptr(), prev_length=sv0["length"].data_ptr(),
                               stats=st, **pg)
                return st.kernel_ms

            def call_chain(st):
                rt.temporal_accumulate_device(None, W, H, a1.data_ptr(), 1, pos, nrm, prm, c1, tcol.data_ptr(),
                                              tln.data_ptr(), prev_color=tp0["color"].data_ptr(),
                                              prev_length=tp0["length"].data_ptr(), stats=st, **pg)
                ms = st.kernel_ms
                rt.denoise_device(None, W, H, tcol.data_ptr(), 1, nrm, pos, alb, prm, dpix.data_ptr(),
                                  dcol.data_ptr(), stats=st)
                return ms + st.kernel_ms

            st = rt.RenderStats()
            for _ in range(3):                                         # warm-up: modules
                call_svgf(st)
                call_chain(st)
            sv, ch = [], []
            for _ in range(a.reps):
                flush.zero_(); torch.cuda.synchronize()
                sv.append(call_svgf(st))
                geo = {k: getattr(st, k) for k in ("launches", "grid", "block")}
                flush.zero_(); torch.cuda.synchronize()
                ch.append(call_chain(st))
            hit = g1["prim"] >= 0
            result["timing"][f"{key}_{W}x{H}"] = {
                "svgf_kernel_ms": {"median": statistics.median(sv), "min": min(sv), "max": max(sv)},
                "chain_kernel_ms": {"median": statistics.median(ch), "min": min(ch), "max": max(ch)},
                "svgf_over_chain": statistics.median(sv) / statistics.median(ch),
                "launch": geo, "hit_fraction": float(hit.float().mean())}
            del a0, g0, sv0, tp0, a1, g1, ill, col, tcol, dcol, mom, ln, tln, pix, dpix
        # quality along the path at 1920x1080, and the sweep on the same frames
        W, H = 1920, 1080
        h = rt.load_world(text)
        frames = []
        for i in range(FRAMES):
            if i:
                rt.move_camera_position(h, *STEP)
            ref = frame(h, W, H, 1024, sample_begin=100_000) / 1024.0
            frames.append((frame(h, W, H, 4, 4 * i), guides(h, W, H), h.camera_floats(), ref))

        def run_svgf(opts):
            prev, ratios = None, []
            for accum, g, cam, ref in frames:
                out = rt.svgf(accum, 4, g, cam, prev, opts)
                hit = g["prim"] >= 0
                ratios.append(mse(out["color"], ref, hit) / mse(accum / 4.0, ref, hit))
                prev = {"camera": cam, "guides": g, "illum": out["illum"], "moments": out["moments"],
                        "length": out["length"]}
            return ratios

        def run_chain():
            prev, ratios = None, []
            for accum, g, cam, ref in frames:
                out = rt.temporal_accumulate(accum, 4, g, cam, prev, pixels=False)
                den = rt.denoise(out["color"], 1, g)
                hit = g["prim"] >= 0
                ratios.append(mse(den["color"], ref, hit) / mse(accum / 4.0, ref, hit))
                prev = {"camera": cam, "guides": g, "color": out["color"], "length": out["length"]}
            return ratios

        result["quality"][key] = {"svgf_ratio_per_frame": run_svgf(rt.SvgfOptions()),
                                  "chain_ratio_per_frame": run_chain()}
        sweep = []
        for sl, mh in itertools.product(SWEEP_SIGMA_LUMINANCE, SWEEP_MAX_HISTORY):
            r = run_svgf(rt.SvgfOptions(sigma_luminance=sl, max_history=mh))
            sweep.append({"sigma_luminance": sl, "max_history": mh, "ratio_per_frame": r,
                          "ratio_max_2_7": max(r[2:]), "ratio_last": r[-1]})
        result["sweep"][key] = sweep
        del frames
    line = json.dumps(result)
    print(line, flush=True)
    if a.out:
        Path(a.out).mkdir(parents=True, exist_ok=True)
        (Path(a.out) / "svgf_bench.json").write_text(line + "\n")


if __name__ == "__main__":
    main()
