"""First-hit buffers against the render of the same primary rays, on one GPU.

    python scripts/aov_bench.py [--reps 20] [--width 3840 --height 2160] [--out DIR]

For the C3 and C5 worlds: the kernel time of render_aov_device (all five buffers) and of render_device with
spp = 1, depth = 1, fixed jitter (one World::hit per pixel on the same camera rays, plus the shading step and the RGBA8
pack), both from the library's CUDA events (RenderStats.kernel_ms).  The two calls alternate, --reps times each, with the
L2 flushed (256 MiB write) between calls; medians, min and max are reported with the card's name and power limit.
Prints one JSON line; --out DIR also writes it to DIR/aov_bench.json.
"""
from __future__ import annotations

import argparse
import importlib
import json
import statistics
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))


def card() -> str:
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--width", type=int, default=3840)
    ap.add_argument("--height", type=int, default=2160)
    ap.add_argument("--worlds", default="c3,c5")
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    import torch
    rt = importlib.import_module("rust-swift-raytracer_b200")
    scenes = importlib.import_module("rust-swift-raytracer_b200.scenes")
    if rt.device_count() < 1:
        raise SystemExit("aov_bench needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    W, H = a.width, a.height
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)        # > 126 MB L2
    bufs = {"depth": torch.empty((H, W), dtype=torch.float32, device=dev),
            "position": torch.empty((H, W, 3), dtype=torch.float32, device=dev),
            "normal": torch.empty((H, W, 3), dtype=torch.float32, device=dev),
            "albedo": torch.empty((H, W, 3), dtype=torch.float32, device=dev),
            "prim": torch.empty((H, W), dtype=torch.int32, device=dev)}
    frame = torch.empty((H, W), dtype=torch.int32, device=dev)
    ptrs = [bufs[k].data_ptr() for k in ("depth", "position", "normal", "albedo", "prim")]
    opt = rt.Options(samples_per_pixel=1, max_ray_bounces=1, fixed_jitter=True, device=0)
    result = {"card": card(), "width": W, "height": H, "reps": a.reps,
              "l2": "flushed between calls (256 MiB write)", "worlds": {}}
    for key in a.worlds.split(","):
        h = rt.load_world(getattr(scenes, key + "_world")())
        st = rt.RenderStats()
        for _ in range(3):                                             # warm-up: modules, scene upload, occupancy
            rt.render_aov_device(h, opt, W, H, *ptrs, stats=st)
            rt.render_device(h, opt, W, H, frame.data_ptr(), stats=st)
        aov, ren = [], []
        for _ in range(a.reps):
            flush.zero_(); torch.cuda.synchronize()
            rt.render_aov_device(h, opt, W, H, *ptrs, stats=st)
            aov.append(st.kernel_ms)
            geo = {k: getattr(st, k) for k in ("grid", "block", "resident", "smem_bytes", "filtered", "culled")}
            flush.zero_(); torch.cuda.synchronize()
            rt.render_device(h, opt, W, H, frame.data_ptr(), stats=st)
            ren.append(st.kernel_ms)
        ma, mr = statistics.median(aov), statistics.median(ren)
        result["worlds"][key] = {
            "aov_kernel_ms": {"median": ma, "min": min(aov), "max": max(aov)},
            "render_spp1_depth1_kernel_ms": {"median": mr, "min": min(ren), "max": max(ren)},
            "ratio_of_medians": ma / mr, "aov_launch": geo,
            "aov_write_gb_per_s": W * H * 44 / (ma * 1e-3) / 1e9}
    line = json.dumps(result)
    print(line, flush=True)
    if a.out:
        Path(a.out).mkdir(parents=True, exist_ok=True)
        (Path(a.out) / "aov_bench.json").write_text(line + "\n")


if __name__ == "__main__":
    main()
