"""Temporal accumulation timing, quality along a camera path, and the sweep that chose its defaults, on one GPU.

    python scripts/temporal_bench.py [--reps 20] [--out DIR]

Timing: for the default world (C2's world and camera) and C3, at 1920x1080 and 3840x2160, the kernel time of
rt_temporal_accumulate_device with default options on a frame whose camera moved since the previous one (the
reprojection path; RenderStats.kernel_ms, CUDA events) alternated with a 1-spp render_device of the same frame, --reps
times each, with the L2 flushed (256 MiB write) before each call; median, min and max, with the card's name and power
limit read in the same run.  The DRAM bytes the call needs at least are counted from the shapes (`min_bytes`).

Quality: along a path of 8 frames of 4 spp (the camera moved by move_camera_position between frames, as a WASD key
press does) at 1920x1080, the mean squared error (linear rgb, hit pixels) of each frame's accumulated colour and of its
own 4-spp mean, both against a 1024-spp frame of that frame's camera (a disjoint sample range); the ratio per frame.

Sweep: the last frame's ratio for a grid of normal_cos x plane_tol x max_history on both worlds.
Prints one JSON line; --out DIR also writes it to DIR/temporal_bench.json.
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
SWEEP_NORMAL_COS = (0.8, 0.9, 0.95)
SWEEP_PLANE_TOL = (0.005, 0.02, 0.05)
SWEEP_MAX_HISTORY = (8, 16, 32)


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
        raise SystemExit("temporal_bench needs a CUDA device")
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

    result = {"card": card(), "reps": a.reps, "l2": "flushed before each call (256 MiB write)",
              "defaults": {"max_history": rt.TEMPORAL_DEFAULT_MAX_HISTORY, "normal_cos": rt.TEMPORAL_DEFAULT_NORMAL_COS,
                           "plane_tol": rt.TEMPORAL_DEFAULT_PLANE_TOL},
              "path": {"frames": FRAMES, "spp": 4, "step": STEP}, "timing": {}, "quality": {}, "sweep": {}}
    for key in a.worlds.split(","):
        text = getattr(scenes, key + "_world")()
        for size in a.sizes.split(","):
            W, H = map(int, size.split("x"))
            h = rt.load_world(text)
            a0, g0, c0 = frame(h, W, H, 1), guides(h, W, H), h.camera_floats()
            prev = rt.temporal_accumulate(a0, 1, g0, c0)
            rt.move_camera_position(h, *STEP)
            a1, g1, c1 = frame(h, W, H, 1, 1), guides(h, W, H), h.camera_floats()
            col = torch.empty((H, W, 4), dtype=torch.float32, device=dev)
            ln = torch.empty((H, W), dtype=torch.float32, device=dev)
            pix = torch.empty((H, W, 4), dtype=torch.uint8, device=dev)
            rpx = torch.empty((H, W), dtype=torch.int32, device=dev)
            args = (None, W, H, a1.data_ptr(), 1, g1["position"].data_ptr(), g1["normal"].data_ptr(),
                    g1["prim"].data_ptr(), c1, col.data_ptr(), ln.data_ptr(), pix.data_ptr())
            hist = dict(prev_camera=c0, prev_position=g0["position"].data_ptr(), prev_normal=g0["normal"].data_ptr(),
                        prev_prim=g0["prim"].data_ptr(), prev_color=prev["color"].data_ptr(),
                        prev_length=prev["length"].data_ptr())
            ropt = rt.Options(samples_per_pixel=1, device=0)
            st = rt.RenderStats()
            for _ in range(3):                                         # warm-up: modules, scene upload
                rt.temporal_accumulate_device(*args, **hist, stats=st)
                rt.render_device(h, ropt, W, H, rpx.data_ptr(), stats=st)
            tem, ren = [], []
            for _ in range(a.reps):
                flush.zero_(); torch.cuda.synchronize()
                rt.temporal_accumulate_device(*args, **hist, stats=st)
                tem.append(st.kernel_ms)
                geo = {k: getattr(st, k) for k in ("launches", "grid", "block")}
                flush.zero_(); torch.cuda.synchronize()
                rt.render_device(h, ropt, W, H, rpx.data_ptr(), stats=st)
                ren.append(st.kernel_ms)
            hit = g1["prim"] >= 0
            kept = float(((ln > 1) & hit).float().sum() / hit.float().sum())
            # at least: this frame's sums (16 B), guides (28 B); the history at hit pixels (4 taps of prev prim, and of
            # normal, position, colour and length where accepted: 48 B per pixel when the taps are mostly shared with
            # the neighbours); colour, length and RGBA8 out (24 B)
            min_bytes = W * H * (16 + 28 + 24) + int(hit.sum()) * 48
            md = statistics.median(tem)
            result["timing"][f"{key}_{W}x{H}"] = {
                "temporal_kernel_ms": {"median": md, "min": min(tem), "max": max(tem)},
                "render_1spp_kernel_ms": {"median": statistics.median(ren), "min": min(ren), "max": max(ren)},
                "launch": geo, "hit_fraction": float(hit.float().mean()), "history_kept_fraction_of_hits": kept,
                "min_bytes": min_bytes, "min_bytes_per_s_at_median": min_bytes / (md * 1e-3)}
            del a0, g0, prev, a1, g1, col, ln, pix, rpx
        # quality along the path at 1920x1080, and the sweep on the same frames
        W, H = 1920, 1080
        h = rt.load_world(text)
        frames = []
        for i in range(FRAMES):
            if i:
                rt.move_camera_position(h, *STEP)
            ref = frame(h, W, H, 1024, sample_begin=100_000) / 1024.0
            frames.append((frame(h, W, H, 4, 4 * i), guides(h, W, H), h.camera_floats(), ref))

        def run(opts):
            prev, ratios = None, []
            for accum, g, cam, ref in frames:
                out = rt.temporal_accumulate(accum, 4, g, cam, prev, opts, pixels=False)
                hit = g["prim"] >= 0
                ratios.append(mse(out["color"], ref, hit) / mse(accum / 4.0, ref, hit))
                prev = {"camera": cam, "guides": g, "color": out["color"], "length": out["length"]}
            return ratios

        result["quality"][key] = {"ratio_per_frame": run(rt.TemporalOptions())}
        sweep = []
        for nc, pt, mh in itertools.product(SWEEP_NORMAL_COS, SWEEP_PLANE_TOL, SWEEP_MAX_HISTORY):
            r = run(rt.TemporalOptions(max_history=mh, normal_cos=nc, plane_tol=pt))
            sweep.append({"normal_cos": nc, "plane_tol": pt, "max_history": mh, "ratio_last": r[-1],
                          "ratio_mean": statistics.mean(r[1:])})
        result["sweep"][key] = sweep
        result["quality"][key]["best_in_sweep"] = min(sweep, key=lambda r: r["ratio_last"])
        del frames
    line = json.dumps(result)
    print(line, flush=True)
    if a.out:
        Path(a.out).mkdir(parents=True, exist_ok=True)
        (Path(a.out) / "temporal_bench.json").write_text(line + "\n")


if __name__ == "__main__":
    main()
