"""Denoiser timing, quality and the sigma sweep that chose its defaults, on one GPU.

    python scripts/denoise_bench.py [--reps 20] [--out DIR]

Timing: for the default world (C2's world and camera) and C3, at 1920x1080 and 3840x2160, the kernel time of
rt_denoise_device with default options (all launches of one call, from the library's CUDA events, RenderStats.kernel_ms)
alternated with a 16-spp render_device of the same frame, --reps times each, with the L2 flushed (256 MiB write)
between calls; median, min and max, with the card's name and power limit read in the same run.

Quality: mean squared error (linear rgb, hit pixels) of the 4-spp frame and of its denoised version, both against a
1024-spp frame of the same world (a different sample range), at 1920x1080.

Sweep: the same error ratio for a grid of sigma_color x sigma_normal x sigma_plane on both worlds at 4 spp.
Prints one JSON line; --out DIR also writes it to DIR/denoise_bench.json.
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

SWEEP_COLOR = (0.25, 0.5, 1.0, 2.0)
SWEEP_NORMAL = (0.25, 0.5, 1.0)
SWEEP_PLANE = (0.02, 0.05, 0.2)


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
        raise SystemExit("denoise_bench needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)        # > 126 MB L2

    def inputs(h, W, H, spp, sample_begin=0):
        accum = torch.empty((H, W, 4), dtype=torch.float32, device=dev)
        frame = torch.empty((H, W), dtype=torch.int32, device=dev)
        rt.render_device(h, rt.Options(samples_per_pixel=spp, accum_out=True, sample_begin=sample_begin, device=0),
                         W, H, frame.data_ptr(), accum.data_ptr())
        torch.cuda.synchronize()
        return accum, frame

    def mse(color, ref, hit):
        d = (color[..., :3].double() - ref[..., :3].double())[hit]
        return float((d * d).mean())

    result = {"card": card(), "reps": a.reps, "l2": "flushed between calls (256 MiB write)",
              "defaults": {"iterations": rt.DENOISE_DEFAULT_ITERATIONS, "sigma_color": rt.DENOISE_DEFAULT_SIGMA_COLOR,
                           "sigma_normal": rt.DENOISE_DEFAULT_SIGMA_NORMAL, "sigma_plane": rt.DENOISE_DEFAULT_SIGMA_PLANE},
              "timing": {}, "quality": {}, "sweep": {}}
    for key in a.worlds.split(","):
        h = rt.load_world(getattr(scenes, key + "_world")())
        for size in a.sizes.split(","):
            W, H = map(int, size.split("x"))
            accum, frame = inputs(h, W, H, 4)
            g = rt.render_aov(h, W, H, rt.Options(fixed_jitter=True, device=0))
            gp = [g[k].data_ptr() for k in ("normal", "position", "albedo", "prim")]
            px = torch.empty((H, W), dtype=torch.int32, device=dev)
            col = torch.empty((H, W, 4), dtype=torch.float32, device=dev)
            ropt = rt.Options(samples_per_pixel=16, device=0)
            st = rt.RenderStats()
            for _ in range(3):                                         # warm-up: modules, scratch, scene upload
                rt.denoise_device(None, W, H, accum.data_ptr(), 4, *gp, px.data_ptr(), col.data_ptr(), stats=st)
                rt.render_device(h, ropt, W, H, frame.data_ptr(), stats=st)
            den, ren = [], []
            for _ in range(a.reps):
                flush.zero_(); torch.cuda.synchronize()
                rt.denoise_device(None, W, H, accum.data_ptr(), 4, *gp, px.data_ptr(), col.data_ptr(), stats=st)
                den.append(st.kernel_ms)
                geo = {k: getattr(st, k) for k in ("launches", "grid", "block")}
                flush.zero_(); torch.cuda.synchronize()
                rt.render_device(h, ropt, W, H, frame.data_ptr(), stats=st)
                ren.append(st.kernel_ms)
            md = statistics.median(den)
            result["timing"][f"{key}_{W}x{H}"] = {
                "denoise_kernel_ms": {"median": md, "min": min(den), "max": max(den)},
                "render_16spp_kernel_ms": {"median": statistics.median(ren), "min": min(ren), "max": max(ren)},
                "denoise_launch": geo,
                "hit_fraction": float((g["prim"] >= 0).float().mean()),
                "ms_per_iteration": md / rt.DENOISE_DEFAULT_ITERATIONS}
            del g, px, col, accum, frame
        # quality and sweep at 1920x1080, 4 spp against 1024 spp (samples 4..1027, independent of the 4-spp frame)
        W, H = 1920, 1080
        accum, _ = inputs(h, W, H, 4)
        ref, _ = inputs(h, W, H, 1024, sample_begin=4)
        ref = ref / 1024.0
        g = rt.render_aov(h, W, H, rt.Options(fixed_jitter=True, device=0))
        hit = g["prim"] >= 0
        e_noisy = mse(accum / 4.0, ref, hit)
        den = rt.denoise(accum, 4, g)
        e_den = mse(den["color"], ref, hit)
        result["quality"][key] = {"mse_noisy_4spp": e_noisy, "mse_denoised": e_den, "ratio": e_den / e_noisy}
        sweep = []
        for sc, sn, sp in itertools.product(SWEEP_COLOR, SWEEP_NORMAL, SWEEP_PLANE):
            d = rt.denoise(accum, 4, g, rt.DenoiseOptions(sigma_color=sc, sigma_normal=sn, sigma_plane=sp))
            sweep.append({"sigma_color": sc, "sigma_normal": sn, "sigma_plane": sp,
                          "ratio": mse(d["color"], ref, hit) / e_noisy})
        result["sweep"][key] = sweep
        result["quality"][key]["best_in_sweep"] = min(sweep, key=lambda r: r["ratio"])
        del g, accum, ref
    line = json.dumps(result)
    print(line, flush=True)
    if a.out:
        Path(a.out).mkdir(parents=True, exist_ok=True)
        (Path(a.out) / "denoise_bench.json").write_text(line + "\n")


if __name__ == "__main__":
    main()
