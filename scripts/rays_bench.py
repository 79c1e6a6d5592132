"""Ray queries (rt_trace_rays_device) on one GPU: against the first-hit buffers of the same camera rays, and on
incoherent rays.

    python scripts/rays_bench.py [--reps 20] [--width 3840 --height 2160] [--incoherent 8388608] [--out DIR]

Coherent: for the C3 and C5 worlds, the un-normalised camera vectors of every pixel centre of a fixed-jitter frame,
((llc + u*horizontal) + v*vertical) - origin in float32, in 8x4 sub-tile order (the order rt_aov_kernel walks its
pixels), traced by trace_rays_device, and the same frame by render_aov_device — all five outputs in both.  The outputs
are first checked to be equal bit for bit.  The two calls then alternate, --reps times each, with the L2 flushed
(256 MiB write) between calls; kernel times come from the library's CUDA events (RenderStats.kernel_ms).
Incoherent: --incoherent rays from the C3 frame's first-hit positions in uniformly random directions; Mrays/s of the
kernel median.  The card's name and power limit are read in the same run.  Prints one JSON line; --out DIR also writes
it to DIR/rays_bench.json.
"""
from __future__ import annotations

import argparse
import importlib
import json
import statistics
import subprocess
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
NAMES = ("depth", "position", "normal", "albedo", "prim")


def card() -> str:
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def camera_rays(cam12: np.ndarray, W: int, H: int):
    """float32 [W*H, 8] rays (camera origin, t_max = +inf, the pixel centre's camera vector) in 8x4 sub-tile order, and
    the row-major pixel index of each ray."""
    F = np.float32
    o, llc, h, v = (cam12[3 * k:3 * k + 3].astype(F) for k in range(4))
    assert W % 8 == 0 and H % 4 == 0
    sy, sx, ly, lx = np.meshgrid(np.arange(H // 4), np.arange(W // 8), np.arange(4), np.arange(8), indexing="ij")
    row, col = (sy * 4 + ly).ravel(), (sx * 8 + lx).ravel()               # image row 0 = top
    u = (col.astype(F) + F(0.5)) / F(W - 1)
    vv = ((H - 1 - row).astype(F) + F(0.5)) / F(H - 1)
    p = ((llc[None, :] + h[None, :] * u[:, None]) + v[None, :] * vv[:, None]) - o[None, :]
    rays = np.zeros((W * H, 8), F)
    rays[:, 0:3] = o
    rays[:, 3] = np.inf
    rays[:, 4:7] = p
    return rays, row * W + col


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--width", type=int, default=3840)
    ap.add_argument("--height", type=int, default=2160)
    ap.add_argument("--worlds", default="c3,c5")
    ap.add_argument("--incoherent", type=int, default=1 << 23)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    import torch
    rt = importlib.import_module("rust-swift-raytracer_b200")
    scenes = importlib.import_module("rust-swift-raytracer_b200.scenes")
    if rt.device_count() < 1:
        raise SystemExit("rays_bench needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    W, H = a.width, a.height
    N = W * H
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)        # > 126 MB L2

    def outputs(n, shape2d=None):
        s1, s3 = ((n,), (n, 3)) if shape2d is None else (shape2d, shape2d + (3,))
        return {"depth": torch.empty(s1, dtype=torch.float32, device=dev),
                "position": torch.empty(s3, dtype=torch.float32, device=dev),
                "normal": torch.empty(s3, dtype=torch.float32, device=dev),
                "albedo": torch.empty(s3, dtype=torch.float32, device=dev),
                "prim": torch.empty(s1, dtype=torch.int32, device=dev)}

    aov, hits = outputs(None, (H, W)), outputs(N)
    aov_ptrs, hit_ptrs = [aov[k].data_ptr() for k in NAMES], [hits[k].data_ptr() for k in NAMES]
    opt = rt.Options(fixed_jitter=True, device=0)
    qopt = rt.RayQueryOptions(device=0)
    result = {"card": card(), "width": W, "height": H, "reps": a.reps,
              "l2": "flushed between calls (256 MiB write)", "coherent": {}, "incoherent": {}}
    first_hits = {}
    for key in a.worlds.split(","):
        h = rt.load_world(getattr(scenes, key + "_world")())
        rays_np, pix = camera_rays(h.camera_floats(), W, H)
        rays = torch.from_numpy(rays_np).to(dev)
        pix_t = torch.from_numpy(pix).to(dev)
        torch.cuda.synchronize()      # the library's stream does not wait for torch's: the rays must be in place
        st = rt.RenderStats()
        for _ in range(3):                                             # warm-up: modules, scene upload, occupancy
            rt.render_aov_device(h, opt, W, H, *aov_ptrs, stats=st)
            rt.trace_rays_device(h, qopt, N, rays.data_ptr(), *hit_ptrs, stats=st)
        same = all(torch.equal(aov[k].reshape(N, -1)[pix_t].view(torch.int32).reshape(hits[k].shape),
                               hits[k].view(torch.int32)) for k in NAMES)
        if not same:
            raise SystemExit(f"{key}: the ray-query outputs differ from render_aov's")
        t_aov, t_ray = [], []
        for _ in range(a.reps):
            flush.zero_(); torch.cuda.synchronize()
            rt.trace_rays_device(h, qopt, N, rays.data_ptr(), *hit_ptrs, stats=st)
            t_ray.append(st.kernel_ms)
            geo = {k: getattr(st, k) for k in ("grid", "block", "resident", "smem_bytes", "filtered", "culled")}
            flush.zero_(); torch.cuda.synchronize()
            rt.render_aov_device(h, opt, W, H, *aov_ptrs, stats=st)
            t_aov.append(st.kernel_ms)
        mr, ma = statistics.median(t_ray), statistics.median(t_aov)
        result["coherent"][key] = {
            "outputs_equal": same,
            "rays_kernel_ms": {"median": mr, "min": min(t_ray), "max": max(t_ray)},
            "aov_kernel_ms": {"median": ma, "min": min(t_aov), "max": max(t_aov)},
            "ratio_of_medians": mr / ma, "rays_launch": geo}
        if key == "c3":
            first_hits[key] = (h, aov["position"][aov["prim"] >= 0].clone())
        del rays, pix_t
    if a.incoherent and "c3" in first_hits:
        h, pos = first_hits["c3"]
        n = a.incoherent
        g = torch.Generator(device=dev).manual_seed(1234)
        idx = torch.randint(0, pos.shape[0], (n,), device=dev, generator=g)
        d = torch.randn((n, 3), device=dev, generator=g)
        rays = torch.zeros((n, 8), dtype=torch.float32, device=dev)
        rays[:, 0:3] = pos[idx]
        rays[:, 3] = float("inf")
        rays[:, 4:7] = d
        torch.cuda.synchronize()      # packed on torch's stream; the calls below run on the library's
        out = outputs(n)
        ptrs = [out[k].data_ptr() for k in NAMES]
        st = rt.RenderStats()
        for _ in range(3):
            rt.trace_rays_device(h, qopt, n, rays.data_ptr(), *ptrs, stats=st)
        ts = []
        for _ in range(a.reps):
            flush.zero_(); torch.cuda.synchronize()
            rt.trace_rays_device(h, qopt, n, rays.data_ptr(), *ptrs, stats=st)
            ts.append(st.kernel_ms)
        m = statistics.median(ts)
        result["incoherent"]["c3"] = {"rays": n, "kernel_ms": {"median": m, "min": min(ts), "max": max(ts)},
                                      "mrays_per_s": n / (m * 1e-3) / 1e6,
                                      "hit_fraction": float((out["prim"] >= 0).float().mean())}
    line = json.dumps(result)
    print(line, flush=True)
    if a.out:
        Path(a.out).mkdir(parents=True, exist_ok=True)
        (Path(a.out) / "rays_bench.json").write_text(line + "\n")


if __name__ == "__main__":
    main()
